"""v210 (WM_PACKED_V210: 10-bit 4:2:2 in 16-byte groups of 6 pixels) through the embed and detect entry points, the host forms, the video
driver and the C++ façade.

The reference is the WM_Y10 path on the same luma samples: `a`, the correlation and the statuses must be its results bit for bit, and every
output luma its output sample.  Every other bit of a row's pitch (chroma, bits 30-31, the unused luma fields of a partial last group, pad
groups) is seeded random in the input and must come through unchanged; bytes past the pitch must not be written.  The v210 packing of this
file's helpers is pinned to the format by a CPU test on a known vector.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import util
from test_gpu_packed_rgb import dev_get, dev_raw, f32bits
from test_gpu_y10 import f32_detect, samples, x_of, y10_path

gpu = pytest.mark.gpu
PSNR = 40.0

# ---- the format: luma of pixel 6g + k in word 4g + WORD[k] at bit BIT[k]; the chroma of pair 3g + j at CB[j] / CR[j] ----
WORD, BIT = (0, 1, 1, 2, 3, 3), (10, 0, 20, 10, 0, 20)
CB, CR = ((0, 0), (1, 10), (2, 20)), ((0, 20), (2, 0), (3, 10))


def pitch(cols):
    return (cols + 47) // 48 * 128


def put(w, wi, bit, v):
    w[:, wi] = (w[:, wi] & ~np.uint32(0x3FF << bit)) | (v.astype(np.uint32) << np.uint32(bit))


def pack(Y, Cb=None, Cr=None, seed=None):
    """(rows, pitch) uint8 v210 rows of luma Y (rows, cols) and chroma Cb / Cr (rows, cols / 2).  seed: every bit that is not a luma sample
    of a pixel (chroma when not given, bits 30-31, unused luma fields of a partial last group, pad groups) is seeded random, else zero."""
    rows, cols = Y.shape
    nw = pitch(cols) // 4
    w = (np.random.default_rng(seed).integers(0, 1 << 32, (rows, nw), dtype=np.uint32) if seed is not None
         else np.zeros((rows, nw), np.uint32))
    for p in range(cols):
        g, k = divmod(p, 6)
        put(w, 4 * g + WORD[k], BIT[k], Y[:, p])
    for c in range(cols // 2):
        g, j = divmod(c, 3)
        for chroma, pos in ((Cb, CB), (Cr, CR)):
            if chroma is not None:
                put(w, 4 * g + pos[j][0], pos[j][1], chroma[:, c])
    return np.ascontiguousarray(w.astype("<u4")).view(np.uint8)


def luma_fields(cols):
    """(word index, bit) of the luma of each pixel of a row"""
    return [(4 * (p // 6) + WORD[p % 6], BIT[p % 6]) for p in range(cols)]


def unpack_luma(b, cols):
    """luma (rows, cols) of v210 rows b (rows, >= pitch) uint8"""
    w = np.ascontiguousarray(b[:, :pitch(cols)]).view("<u4")
    return np.stack([(w[:, wi] >> np.uint32(bit)) & 0x3FF for wi, bit in luma_fields(cols)], axis=1).astype(np.uint16)


def luma_bits(cols):
    """(pitch / 4,) uint32 mask of the bits of a row that are the luma of its pixels"""
    m = np.zeros(pitch(cols) // 4, np.uint32)
    for wi, bit in luma_fields(cols):
        m[wi] |= np.uint32(0x3FF << bit)
    return m


def non_luma(b, cols):
    return np.ascontiguousarray(b[..., :pitch(cols)]).view("<u4") & ~luma_bits(cols)


def test_pack_matches_the_format():
    """the helpers against the format's known vector, without the library"""
    Y = np.array([[64, 940, 512, 1, 1023, 300]], np.uint16)
    got = pack(Y, np.array([[100, 200, 300]]), np.array([[400, 500, 600]]))
    assert [int(x) for x in got[0, :16].view("<u4")] == [0x19010064, 0x200323AC, 0x12C005F4, 0x12C963FF]
    assert bytes(got[0, :16]) == bytes.fromhex("64000119ac230320f405c012ff63c912")
    assert np.all(got[0, 16:] == 0) and got.shape == (1, 128)
    assert np.array_equal(unpack_luma(got, 6), Y)
    assert [pitch(c) for c in (1920, 3840, 1280)] == [5120, 10240, 3456]
    r = pack(samples(5, 202, seed=1), seed=3)
    assert np.array_equal(unpack_luma(r, 202), samples(5, 202, seed=1))


# ---- the library ----
def wm_for(wmb, rows, cols, p, W=None):
    return wmb.Watermark(rows, cols, util.normal_w(rows, cols) if W is None else W, p, PSNR)


def place(imgs, ld, stride, fill):
    """v210 images (batch, rows, pitch) into one buffer: rows `ld` bytes apart, images `stride` bytes apart, `fill` elsewhere"""
    batch, rows, pb = imgs.shape
    buf = np.full(batch * stride, fill, np.uint8)
    for b in range(batch):
        buf[b * stride:b * stride + rows * ld].reshape(rows, ld)[:, :pb] = imgs[b]
    return buf


def take(buf, batch, rows, pb, ld, stride):
    return np.stack([buf[b * stride:b * stride + rows * ld].reshape(rows, ld)[:, :pb] for b in range(batch)])


def v210_path(wmb, wm, imgs, cols, mask, ld=0, stride=0):
    """wm_embed_batch (base = in) and wm_detect_batch on the input and on the output of v210 images (batch, rows, pitch) placed at a row
    pitch of `ld` bytes and a batch stride of `stride` bytes -> (out (batch, rows, pitch), a, status, corr of in, status, corr of out, status).
    Checks that the input is only read and that no output byte past a row's pitch is written."""
    batch, rows, pb = imgs.shape
    ldb = ld or pb
    sb = stride or rows * ldb
    buf = place(imgs, ldb, sb, 0x5C)
    pin, pout = dev_raw(wmb, wm, buf), dev_raw(wmb, wm, np.full(buf.shape, 0xA5, np.uint8))
    desc = lambda p: wmb.image_desc(p, rows, cols, wmb.PACKED_V210, wmb.U8, ld, 0)
    a, st = np.full(batch, np.nan, np.float32), np.zeros(batch, np.int32)
    ci, sti, co, sto = np.zeros(batch, np.float32), np.zeros(batch, np.int32), np.zeros(batch, np.float32), np.zeros(batch, np.int32)
    wm.embed_batch(0, desc(pin), desc(pin), desc(pout), stride, stride, stride, batch, mask, a, st)
    wm.detect_batch(0, desc(pin), stride, batch, mask, ci, sti)
    wm.detect_batch(0, desc(pout), stride, batch, mask, co, sto)
    wm.sync(0)
    ob = dev_get(wmb, wm, pout, buf.shape)
    assert np.array_equal(dev_get(wmb, wm, pin, buf.shape), buf)
    for p in (pin, pout):
        wmb.lib().wm_dev_free(wm._h, p)
    written = place(np.ones(imgs.shape, np.uint8), ldb, sb, 0).astype(bool)
    assert np.all(ob[~written] == 0xA5)  # nothing past the pitch, nothing between images
    return take(ob, batch, rows, pb, ldb, sb), a, st, ci, sti, co, sto


def assert_equal_to_y10(wmb, wm, v, mask, ld=0, stride=0, seed=0, what=""):
    """v210 images of luma v (batch, rows, cols), all other bits random, against WM_Y10 on words holding v"""
    batch, rows, cols = v.shape
    imgs = np.stack([pack(v[b], seed=seed + b) for b in range(batch)])
    out, a, st, ci, sti, co, sto = v210_path(wmb, wm, imgs, cols, mask, ld, stride)
    ref = y10_path(wmb, wm, v, wmb.Y10, mask)
    print("%s: a=%r corr(in)=%r corr(out)=%r status=%r" % (what, a[0], ci[0], co[0], st[0]))
    for got, r in zip((a, ci, co), (ref[1], ref[3], ref[5])):
        assert np.array_equal(got.view(np.uint32), r.view(np.uint32)), what
    assert np.array_equal(st, ref[2]) and np.array_equal(sti, ref[4]) and np.array_equal(sto, ref[6]), what
    for b in range(batch):
        assert np.array_equal(unpack_luma(out[b], cols), ref[0][b]), (what, b)
    assert np.array_equal(non_luma(out, cols), non_luma(imgs, cols)), what  # every other bit of the pitch is the input's
    return out, a, st


CASES = [(0, 3), (1, 3), (1, 7)]  # (mask, p): ME, NVF 3x3, NVF 7x7


@gpu
@pytest.mark.parametrize("rows,cols", [(1080, 1920), (121, 1280), (67, 202), (9, 4), (9, 6)])
def test_equal_to_y10(wmb, rows, cols):
    """1920 and 1280 columns: cols % 6 = 0 and 2, the latter with pad groups; 202: cols % 6 = 4; 4 and 6: a single group"""
    v = samples(rows, cols, seed=rows + cols)
    for mask, p in CASES:
        wm = wm_for(wmb, rows, cols, p)
        assert_equal_to_y10(wmb, wm, v[None], mask, seed=cols, what="%dx%d mask=%d p=%d" % (rows, cols, mask, p))
        wm.close()


@gpu
@pytest.mark.parametrize("rows,cols", [(1080, 1920), (121, 1280), (67, 202)])
def test_padded_rows_and_strided_batch(wmb, rows, cols):
    """rows 64 bytes (16-aligned) and 4 bytes (word- but not 16-aligned) past the pitch; a batch of 3 at a stride larger than one image"""
    vs = np.stack([samples(rows, cols, seed=40 + b) for b in range(3)])
    for mask, p in CASES:
        wm = wm_for(wmb, rows, cols, p)
        what = "%dx%d mask=%d p=%d" % (rows, cols, mask, p)
        for extra in (64, 4):
            ld = pitch(cols) + extra
            assert_equal_to_y10(wmb, wm, vs[:1], mask, ld=ld, seed=extra, what="ld+%d %s" % (extra, what))
            assert_equal_to_y10(wmb, wm, vs, mask, ld=ld, stride=rows * ld + 36, seed=extra, what="batch 3 ld+%d %s" % (extra, what))
        wm.close()


@gpu
def test_against_oracle(wmb, oracle):
    rows, cols = 512, 512
    v = samples(rows, cols, seed=5)
    x = x_of(v)
    W = util.normal_w(rows, cols)
    wm = wm_for(wmb, rows, cols, 3, W)
    for mask in (wmb.ME, wmb.NVF):
        o = oracle.embed(x, W, PSNR, mask)
        out, a, st, ci, sti, co, sto = v210_path(wmb, wm, pack(v, seed=5)[None], cols, mask)
        got = unpack_luma(out[0], cols)
        dv = int(np.abs(got.astype(np.int64) - np.clip(4.0 * np.asarray(o["out"], np.float64), 0, 1023).astype(np.int64)).max())
        od, di = oracle.detect(x_of(got), W, mask), oracle.detect(x, W, mask)
        ra, rc, ri = util.rel(a[0], o["a"]), util.rel(co[0], od["corr"]), util.rel(ci[0], di["corr"])
        print("oracle mask=%d: a rel %.3g corr(out) rel %.3g corr(in) rel %.3g max sample diff %d" % (mask, ra, rc, ri, dv))
        assert st[0] == 0 and sto[0] == 0 and sti[0] == 0
        assert ra <= 1e-3 and rc <= 1e-3 and ri <= 1e-3 and dv <= 1
    wm.close()


@gpu
def test_singular_and_zero_mask(wmb):
    rows, cols = 121, 1280
    wm = wm_for(wmb, rows, cols, 3)
    wz = wm_for(wmb, rows, cols, 3, np.zeros((rows, cols), np.float32))
    img = pack(np.full((rows, cols), 469, np.uint16), seed=1)[None]  # constant luma: the ME system is unsolvable
    out, a, st, *_ = v210_path(wmb, wm, img, cols, wmb.ME)
    assert st[0] == wmb.SINGULAR and np.isnan(a[0]) and np.array_equal(out, img)
    img = pack(samples(rows, cols, seed=8), seed=2)[None]
    for mask in (wmb.ME, wmb.NVF):
        out, a, st, *_ = v210_path(wmb, wz, img, cols, mask)
        assert st[0] == wmb.ZERO_MASK and np.isinf(a[0]) and np.array_equal(out, img), mask
    wz.close()
    wm.close()


@gpu
@pytest.mark.parametrize("cols,extra", [(1920, 0), (1280, 0), (202, 4), (6, 12)])
def test_rows_ending_at_the_allocation_end(wmb, cols, extra):
    """the last row of in and out ends at the last byte of its allocation: nothing past the pitch is read or written"""
    rows = 31
    pb = pitch(cols)
    ld = pb + extra
    v = samples(rows, cols, seed=cols)
    img = pack(v, seed=cols)
    n = (rows - 1) * ld + pb
    buf = place(img[None], ld, rows * ld, 0)[:n]
    wm = wm_for(wmb, rows, cols, 3)
    L = wmb.lib()
    for mask in (wmb.ME, wmb.NVF):
        ref = y10_path(wmb, wm, v[None], wmb.Y10, mask)
        pin, pout = dev_raw(wmb, wm, buf), dev_raw(wmb, wm, np.zeros_like(buf))
        desc = lambda p: wmb.image_desc(p, rows, cols, wmb.PACKED_V210, wmb.U8, ld, 0)
        a, st, corr, st2 = np.full(1, np.nan, np.float32), np.zeros(1, np.int32), np.zeros(1, np.float32), np.zeros(1, np.int32)
        wm.embed_batch(0, desc(pin), desc(pin), desc(pout), 0, 0, 0, 1, mask, a, st)
        wm.detect_batch(0, desc(pin), 0, 1, mask, corr, st2)
        wm.sync(0)
        o = np.concatenate([dev_get(wmb, wm, pout, buf.shape), np.zeros(rows * ld - n, np.uint8)])
        for p in (pin, pout):
            L.wm_dev_free(wm._h, p)
        got = o.reshape(rows, ld)[:, :pb]
        assert np.array_equal(unpack_luma(got, cols), ref[0][0]) and np.array_equal(non_luma(got, cols), non_luma(img, cols))
        assert st[0] == ref[2][0] and f32bits(a[0]) == f32bits(ref[1][0]) and f32bits(corr[0]) == f32bits(ref[3][0])
    wm.close()


@gpu
@pytest.mark.parametrize("rows,cols", [(121, 1280), (1080, 1920)])
def test_synchronous_embed_after_replay(wmb, rows, cols):
    """wm_embed with the same arguments again and again is captured into a CUDA graph and replayed; its output must be complete when it
    returns, every time: the pack kernel, the op's last, publishes the result"""
    img = pack(samples(rows, cols, seed=12), seed=12)
    wm = wm_for(wmb, rows, cols, 3)
    ref, ra, rst, *_ = v210_path(wmb, wm, img[None], cols, wmb.ME)
    d = wmb.DeviceArray.from_numpy(wm, img, wmb.PACKED_V210)
    o = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_V210)
    for it in range(6):  # the same arguments every time: captured on the second call, replayed from the third
        o.upload(np.zeros_like(img))
        _, a, st = wm.makeWatermark(d, None, wmb.ME, out=o)
        got = o.numpy()
        assert np.array_equal(got, ref[0]), (it, int(np.count_nonzero(got != ref[0])))
        assert st == rst[0] and f32bits(a) == f32bits(ra[0]), it
    o.free()
    for it in range(4):
        corr, st = wm.detectWatermark(d, wmb.ME)
        assert st == 0
    d.free()
    wm.close()


@gpu
def test_host_forms_equal_device_forms(wmb):
    rows, cols, batch = 67, 202, 3
    pb = pitch(cols)
    wm = wm_for(wmb, rows, cols, 3)
    L = wmb.lib()
    imgs = np.stack([pack(samples(rows, cols, seed=60 + b), seed=60 + b) for b in range(batch)])
    for mask in (wmb.ME, wmb.NVF):
        refs = [v210_path(wmb, wm, imgs[b:b + 1], cols, mask) for b in range(batch)]
        big = np.zeros((rows, pb + 64), np.uint8)  # rows of a pitched host buffer
        big[:, :pb] = imgs[0]
        out = np.full((rows, pb + 64), 0x3C, np.uint8)
        a, st = wm.make_watermark_host(big[:, :pb], None, out[:, :pb], mask, layout=wmb.PACKED_V210)
        corr, st2 = wm.detect_watermark_host(big[:, :pb], mask, layout=wmb.PACKED_V210)
        assert np.array_equal(out[:, :pb], refs[0][0][0]) and np.all(out[:, pb:] == 0x3C)
        assert f32bits(a) == f32bits(refs[0][1][0]) and st == refs[0][2][0]
        assert f32bits(corr) == f32bits(refs[0][3][0]) and st2 == refs[0][4][0]
        nb = rows * pb
        hp = [L.wm_host_alloc_pinned(batch * nb) for _ in range(2)]
        hin, hout = [np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), (batch, rows, pb)) for p in hp]
        hin[:] = imgs
        desc = lambda p: wmb.image_desc(p, rows, cols, wmb.PACKED_V210, wmb.U8, 0, 0)
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
            assert f32bits(corr[b]) == f32bits(refs[b][5][0])  # detection on the written words
        corr[:] = 0
        wm.detect_host_batch(3, desc(hp[0]), 0, batch, mask, corr, st2)
        wm.sync(3)
        for b in range(batch):
            assert f32bits(corr[b]) == f32bits(refs[b][3][0]) and st2[b] == refs[b][4][0]
        for p in hp:
            L.wm_host_free_pinned(p)
    wm.close()


# ---- the video driver ----
VROWS, VCOLS = 270, 480  # 36 tiles: a frame's partial sums are grouped the same way whatever run it shares


def video_frames(n, seed=0):
    return np.stack([pack(np.roll(samples(VROWS, VCOLS, seed=seed + i % 3), 11 * i, axis=1), seed=seed + i) for i in range(n)])


def run_driver(wmb, wm, frames, mode, interval, first, on_device, linesize=0, ctxs=None):
    """wm_process_frames (or _multi over `ctxs`) on v210 frames (n, rows, pitch) at a row pitch of `linesize` -> (out (n, rows, pitch), scalars)"""
    n, rows, pb = frames.shape
    ls = linesize or pb
    buf = place(frames, ls, rows * ls, 0x33)
    obytes = rows * pb
    L = wmb.lib()
    embed = mode != wmb.VIDEO_DETECT
    scal = np.full(2 * n if mode == wmb.VIDEO_EMBED_VERIFY else n, 7.0, np.float32)
    if on_device:
        src = dev_raw(wmb, wm, buf)
        dst = dev_raw(wmb, wm, np.full(n * obytes, 0xA5, np.uint8)) if embed else None
    else:
        src, host_out = buf.ctypes.data, np.full((n, obytes), 0xA5, np.uint8)
        dst = host_out.ctypes.data if embed else None
    if ctxs is None:
        v = wmb.VideoProcessingContext(wm, rows, VCOLS, interval, linesize=linesize, frames_on_device=on_device, layout=wmb.PACKED_V210)
        assert wmb.process_frames(v, mode, src, dst, first, n, scal) == n
    else:
        vs = [wmb.VideoProcessingContext(c, rows, VCOLS, interval, linesize=linesize, frames_on_device=on_device, layout=wmb.PACKED_V210)
              for c in ctxs]
        firsts = [wmb.shard_frames(n, g, len(ctxs))[0] for g in range(len(ctxs))]
        assert wmb.process_frames_multi(vs, mode, [src + f * rows * ls for f in firsts], [dst + f * obytes for f in firsts] if embed else None,
                                        first, n, scal) == n
    out = None
    if embed:
        out = (dev_get(wmb, wm, dst, (n, obytes)) if on_device else host_out).reshape(n, rows, pb)
    if on_device:
        L.wm_dev_free(wm._h, src)
        if embed:
            L.wm_dev_free(wm._h, dst)
    return out, scal


@gpu
@pytest.mark.parametrize("on_device", [False, True])
def test_video_driver(wmb, on_device):
    n, first, interval = 10, 2, 3
    pb = pitch(VCOLS)
    wm = wm_for(wmb, VROWS, VCOLS, 3)
    frames = video_frames(n, seed=30)
    gated = (first + np.arange(n)) % interval == 0
    refs = {i: v210_path(wmb, wm, frames[i:i + 1], VCOLS, wmb.ME) for i in range(n) if gated[i]}
    for ls in (0, pb + 64, pb + 4):
        what = "device=%d linesize=%d" % (on_device, ls)
        out, a = run_driver(wmb, wm, frames, wmb.VIDEO_EMBED, interval, first, on_device, linesize=ls)
        _, corr = run_driver(wmb, wm, out, wmb.VIDEO_DETECT, interval, first, on_device)
        o2, s2 = run_driver(wmb, wm, frames, wmb.VIDEO_EMBED_VERIFY, interval, first, on_device, linesize=ls)
        _, cin = run_driver(wmb, wm, frames, wmb.VIDEO_DETECT, interval, first, on_device, linesize=ls)
        assert np.array_equal(o2, out), what
        assert np.all(np.isnan(a[~gated])) and np.all(np.isnan(corr[~gated])) and np.all(np.isnan(s2[n:][~gated])), what
        for i in range(n):
            if not gated[i]:
                assert np.array_equal(out[i], frames[i]), (what, i)  # copied through, every byte of the pitch
                continue
            ro, ra, rst, rci, _, rco, _ = refs[i]
            assert np.array_equal(out[i], ro[0]), (what, i)
            assert f32bits(a[i]) == f32bits(ra[0]) == f32bits(s2[i]), (what, i)
            assert f32bits(corr[i]) == f32bits(rco[0]) == f32bits(s2[n + i]), (what, i)
            assert f32bits(cin[i]) == f32bits(rci[0]), (what, i)
    wm.close()


@gpu
@pytest.mark.parametrize("on_device", [False, True])
def test_video_multi_equals_single(wmb, on_device):
    n, first, interval = 11, 1, 3
    ls = pitch(VCOLS) + 64
    wm = wm_for(wmb, VROWS, VCOLS, 3)
    clones = [wm.clone(), wm.clone()]
    frames = video_frames(n, seed=50)
    o1, a1 = run_driver(wmb, wm, frames, wmb.VIDEO_EMBED, interval, first, on_device, linesize=ls)
    o2, a2 = run_driver(wmb, wm, frames, wmb.VIDEO_EMBED, interval, first, on_device, linesize=ls, ctxs=clones)
    assert np.array_equal(o1, o2) and np.array_equal(a1.view(np.uint32), a2.view(np.uint32))
    _, c1 = run_driver(wmb, wm, o1, wmb.VIDEO_DETECT, interval, first, on_device)
    _, c2 = run_driver(wmb, wm, o1, wmb.VIDEO_DETECT, interval, first, on_device, ctxs=clones)
    assert np.array_equal(c1.view(np.uint32), c2.view(np.uint32))
    for c in clones:
        c.close()
    wm.close()


@gpu
def test_video_rejections(wmb):
    rows, cols, n = 31, 202, 2
    pb = pitch(cols)
    wm = wm_for(wmb, rows, cols, 3)
    frames = np.zeros(n * rows * (pb + 8) + 8, np.uint8)
    out = np.zeros_like(frames)
    scal = np.zeros(2 * n, np.float32)
    for ls, fstride, off in ((pb - 4, 0, 0), (pb + 2, 0, 0), (0, rows * pb + 2, 0), (0, 0, 2)):
        v = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=ls, frame_stride=fstride, layout=wmb.PACKED_V210)
        with pytest.raises(wmb.WatermarkError) as e:
            wmb.process_frames(v, wmb.VIDEO_EMBED, frames.ctypes.data + off, out.ctypes.data, 0, n, scal)
        print("linesize %d frame_stride %d offset %d: %s" % (ls, fstride, off, e.value))
        assert e.value.code == -5
    assert np.all(out == 0)
    wm.close()
    wo = wm_for(wmb, rows, cols + 1, 3)  # odd width
    v = wmb.VideoProcessingContext(wo, rows, cols + 1, 1, layout=wmb.PACKED_V210)
    with pytest.raises(wmb.WatermarkError) as e:
        wmb.process_frames(v, wmb.VIDEO_EMBED, frames.ctypes.data, out.ctypes.data, 0, n, scal)
    assert e.value.code == -5
    wo.close()


@gpu
def test_rejections(wmb):
    rows, cols = 31, 202
    pb = pitch(cols)
    wm = wm_for(wmb, rows, cols, 3)
    L = wmb.lib()
    img = pack(samples(rows, cols), seed=1)
    d = wmb.DeviceArray.from_numpy(wm, img, wmb.PACKED_V210)
    assert np.array_equal(d.numpy(), img)
    out = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_V210)
    y10 = wmb.DeviceArray(wm, rows, cols, wmb.Y10)
    yuyv = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_YUYV)
    gray = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.F32, 1)
    y8 = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.U8, 1)
    big = L.wm_dev_alloc(wm._h, 4 * rows * (pb + 32))
    far = big + 2 * rows * (pb + 32)
    a = C.c_float(0)

    def desc(p, dtype=wmb.U8, ld=0, ch=0, layout=wmb.PACKED_V210):
        return wmb.image_desc(p, rows, cols, layout, dtype, ld, ch)

    def embed_rc(i, b, o):
        return L.wm_embed(wm._h, C.byref(i), C.byref(b) if b is not None else None, C.byref(o), wmb.ME, C.byref(a))

    def detect_rc(i):
        return L.wm_detect(wm._h, C.byref(i), wmb.ME, C.byref(a))

    def refused(rc, what):
        msg = L.wm_last_error(wm._h).decode()
        print("%s: %d %s" % (what, rc, msg))
        assert rc == -5 and msg, what

    refused(embed_rc(desc(d.ptr, dtype=wmb.F32), None, out.desc()), "f32 dtype")
    for ch in (1, 2, 4):
        refused(detect_rc(desc(d.ptr, ch=ch)), "%d channels" % ch)
    refused(embed_rc(desc(d.ptr), None, desc(far, ch=2)), "out with 2 channels")
    refused(detect_rc(desc(big, ld=pb + 2)), "ld not a multiple of 4")
    refused(detect_rc(desc(big, ld=pb - 4)), "ld below the pitch")
    refused(detect_rc(desc(big, ld=2 * cols)), "ld of 2 bytes per pixel")
    refused(detect_rc(desc(big + 2)), "pointer not word-aligned")
    refused(embed_rc(desc(d.ptr), None, desc(far + 2)), "out pointer not word-aligned")
    refused(embed_rc(desc(d.ptr), None, desc(far, ld=pb + 6)), "out ld not a multiple of 4")
    wo = wm_for(wmb, rows, cols + 1, 3)
    rc = L.wm_detect(wo._h, C.byref(wmb.image_desc(big, rows, cols + 1, wmb.PACKED_V210, wmb.U8, 0, 0)), wmb.ME, C.byref(a))
    assert rc == -5, "odd cols"
    wo.close()
    corr, st = np.zeros(2, np.float32), np.zeros(2, np.int32)
    cp, sp = corr.ctypes.data_as(C.POINTER(C.c_float)), st.ctypes.data_as(C.POINTER(C.c_int))
    refused(L.wm_detect_batch(wm._h, 0, C.byref(desc(big)), rows * pb + 2, 2, wmb.ME, cp, sp), "batch stride not a multiple of 4")
    refused(L.wm_embed_batch(wm._h, 0, C.byref(desc(big)), None, C.byref(desc(far)), rows * pb, 0, rows * pb + 6, 2, wmb.ME, cp, sp),
            "out batch stride not a multiple of 4")
    refused(L.wm_rgb2gray(wm._h, C.byref(d.desc()), C.byref(gray.desc()), 0.299, 0.587, 0.114), "rgb2gray")
    refused(L.wm_debug_plane(wm._h, C.byref(d.desc()), wmb.DBG_ERRSEQ, gray.ptr), "debug_plane")
    refused(L.wm_debug_detect_planes(wm._h, C.byref(d.desc()), wmb.ME, gray.ptr, gray.ptr, C.byref(a)), "debug_detect_planes")
    for o, name in ((y10, "Y10"), (yuyv, "YUYV"), (y8, "Y plane"), (gray, "gray")):
        refused(embed_rc(d.desc(), None, o.desc()), "v210 in, %s out" % name)
        refused(embed_rc(o.desc(), None, out.desc()), "%s in, v210 out" % name)
    refused(embed_rc(d.desc(), desc(d.ptr, ch=2, layout=wmb.Y10), out.desc()), "Y10 base")
    refused(embed_rc(d.desc(), y8.desc(), out.desc()), "Y-plane base")
    refused(embed_rc(d.desc(), None, desc(d.ptr + 16)), "out overlaps in")
    # host forms
    h, o = img.copy(), np.zeros_like(img)
    hd = lambda arr, layout=wmb.PACKED_V210, ld=0, ch=0, off=0: wmb.image_desc(arr.ctypes.data + off, rows, cols, layout, wmb.U8, ld, ch)
    refused(L.wm_embed_host(wm._h, C.byref(hd(h)), None, C.byref(hd(o, wmb.Y10, ch=2)), wmb.ME, C.byref(a)), "host v210 in, Y10 out")
    refused(L.wm_detect_host(wm._h, C.byref(hd(h, ld=pb + 2)), wmb.ME, C.byref(a)), "host ld not a multiple of 4")
    refused(L.wm_detect_host(wm._h, C.byref(hd(h, ld=pb - 4)), wmb.ME, C.byref(a)), "host ld below the pitch")
    refused(L.wm_detect_host(wm._h, C.byref(hd(h, ch=2)), wmb.ME, C.byref(a)), "host 2 channels")
    hb = np.zeros(2 * rows * pb + 16, np.uint8)
    refused(L.wm_detect_host_batch(wm._h, 0, C.byref(hd(hb)), rows * pb + 2, 2, wmb.ME, cp, sp), "host batch stride")
    refused(L.wm_detect_host(wm._h, C.byref(hd(hb, off=2)), wmb.ME, C.byref(a)), "host misaligned pointer")
    refused(L.wm_embed_verify_host_batch(wm._h, 0, C.byref(hd(h)), None, C.byref(hd(o, ld=pb + 2)), 0, 0, 0, 1, wmb.ME, cp, cp, sp),
            "embed_verify out ld")
    assert np.all(o == 0)
    with pytest.raises(TypeError):
        wm.make_watermark_host(h[:, :pb - 4], None, o, wmb.ME, layout=wmb.PACKED_V210)
    for x in (d, out, y10, yuyv, gray, y8):
        x.free()
    L.wm_dev_free(wm._h, big)
    wm.close()


@gpu
def test_cpp_process_frames_in_memory_v210(wmb, tmp_path):
    b = wmb.build()
    exe = b.build_video_v210_test()
    assert exe and os.path.exists(exe)
    n, interval = 7, 2
    pb = pitch(VCOLS)
    ls = pb + 64
    W = util.normal_w(VROWS, VCOLS)
    frames = video_frames(n, seed=70)
    place(frames, ls, VROWS * ls, 0x77).tofile(tmp_path / "frames.u8")
    W.tofile(tmp_path / "w.dat")
    r = subprocess.run([exe, str(tmp_path / "w.dat"), str(VROWS), str(VCOLS), str(tmp_path / "frames.u8"), str(n), str(ls), str(interval),
                        str(tmp_path / "out.u8")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = dict(line.split(None, 1) for line in r.stdout.strip().splitlines())
    assert got["frames"].split() == [str(n), str(n)]
    assert got["equal_pixels"].strip() == "1" and got["equal_a"].strip() == "1" and got["nan_where_gated_off"].strip() == "1"
    assert float(got["corr_max_rel"]) == 0.0
    wm = wmb.Watermark(VROWS, VCOLS, W, 3, PSNR)
    out, a = run_driver(wmb, wm, frames, wmb.VIDEO_EMBED, interval, 0, False, linesize=ls)
    _, corr = run_driver(wmb, wm, out, wmb.VIDEO_DETECT, interval, 0, False)
    assert np.array_equal(np.fromfile(tmp_path / "out.u8", np.uint8).reshape(out.shape), out)
    for i in range(n):
        assert np.array_equal(np.float32(got["a_%d" % i]), a[i], equal_nan=True)
        assert np.array_equal(np.float32(got["corr_%d" % i]), corr[i], equal_nan=True)
    wm.close()
