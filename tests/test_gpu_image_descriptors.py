"""Return codes of malformed image descriptors on every entry-point family.

Each call has one fault in a planar descriptor (layout, dtype, channels, ld, batch stride) and gets WM_ERR_ARG, or two faults whose
order decides the code: an image on the device is compared with the watermark's dims before the rest of its descriptor is checked
(WM_ERR_DIMS), a host image after it (WM_ERR_ARG), because its dims are compared on the staged copy.  The video driver checks its mode,
the frame dims, the interval and `out` before the frame descriptor, and takes layout 0 and WM_ROW_MAJOR as the same Y-plane frames.
"""
import ctypes as C

import numpy as np
import pytest

import util
from test_gpu_packed_rgb import dev_get, dev_raw

pytestmark = pytest.mark.gpu

PSNR = 40.0
ROWS, COLS = 67, 130
DIMS, ARG = -4, -5
BATCH = 2
IMAGE = 4 * (ROWS + 1) * (COLS + 1)  # f32 elements of the largest image the calls below describe (four planes, one row and col more)


@pytest.fixture(scope="module")
def env(wmb):
    """a watermark, three device buffers and three host buffers (in, base, out) of BATCH such images each"""
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    zeros = np.zeros(BATCH * IMAGE, np.float32)
    dev = [dev_raw(wmb, wm, zeros) for _ in range(3)]
    host = [zeros.copy() for _ in range(3)]
    yield wm, dev, host
    for p in dev:
        wmb.lib().wm_dev_free(wm._h, p)
    wm.close()


def desc(wmb, ptr, rows=ROWS, cols=COLS, layout=None, dtype=None, ld=0, ch=1, ps=0):
    return wmb.image_desc(ptr, rows, cols, wmb.ROW_MAJOR if layout is None else layout, wmb.F32 if dtype is None else dtype, ld, ch, ps)


def expect(wmb, wm, rc, code, what):
    msg = wmb.lib().wm_last_error(wm._h).decode()
    print("%s: %d %s" % (what, rc, msg))
    assert rc == code and msg, what


# one fault of a planar descriptor, on any image
def planar_faults(wmb):
    return [("layout 99", dict(layout=99)), ("layout -1", dict(layout=-1)), ("dtype 7", dict(dtype=7)), ("ld < cols", dict(ld=COLS - 1)),
            ("col-major ld < rows", dict(layout=wmb.COL_MAJOR, ld=ROWS - 1))]


def embed_forms(wmb, wm):
    """name -> (on the device, call(in, base, out, strides) -> rc)"""
    L = wmb.lib()
    a, corr, st = np.zeros(BATCH, np.float32), np.zeros(BATCH, np.float32), np.zeros(BATCH, np.int32)
    fa, fc, ist = (x.ctypes.data_as(C.POINTER(C.c_float if x.dtype == np.float32 else C.c_int)) for x in (a, corr, st))
    r = C.byref
    return {
        "wm_embed": (True, lambda i, b, o, s: L.wm_embed(wm._h, r(i), r(b), r(o), wmb.ME, fa)),
        "wm_embed_batch": (True, lambda i, b, o, s: L.wm_embed_batch(wm._h, 0, r(i), r(b), r(o), *s, BATCH, wmb.ME, fa, ist)),
        "wm_embed_host": (False, lambda i, b, o, s: L.wm_embed_host(wm._h, r(i), r(b), r(o), wmb.ME, fa)),
        "wm_embed_host_batch": (False, lambda i, b, o, s: L.wm_embed_host_batch(wm._h, 0, r(i), r(b), r(o), *s, BATCH, wmb.ME, fa, ist)),
        "wm_embed_verify_host_batch": (False, lambda i, b, o, s: L.wm_embed_verify_host_batch(wm._h, 0, r(i), r(b), r(o), *s, BATCH, wmb.ME,
                                                                                                fa, fc, ist)),
    }


def detect_forms(wmb, wm):
    """name -> (on the device, call(img, stride) -> rc)"""
    L = wmb.lib()
    corr, st = np.zeros(BATCH, np.float32), np.zeros(BATCH, np.int32)
    fc, ist = corr.ctypes.data_as(C.POINTER(C.c_float)), st.ctypes.data_as(C.POINTER(C.c_int))
    r = C.byref
    return {
        "wm_detect": (True, lambda d, s: L.wm_detect(wm._h, r(d), wmb.ME, fc)),
        "wm_detect_batch": (True, lambda d, s: L.wm_detect_batch(wm._h, 0, r(d), s, BATCH, wmb.ME, fc, ist)),
        "wm_detect_host": (False, lambda d, s: L.wm_detect_host(wm._h, r(d), wmb.ME, fc)),
        "wm_detect_host_batch": (False, lambda d, s: L.wm_detect_host_batch(wm._h, 0, r(d), s, BATCH, wmb.ME, fc, ist)),
    }


def test_embed_planar_faults(wmb, env):
    wm, dev, host = env
    for name, (on_device, call) in embed_forms(wmb, wm).items():
        pi, pb, po = (p if on_device else h.ctypes.data for p, h in zip(dev, host))
        ok = lambda p, **kw: desc(wmb, p, **kw)

        def rc(what, code, i=None, b=None, o=None, s=(0, 0, 0)):
            expect(wmb, wm, call(i or ok(pi), b or ok(pi), o or ok(po), s), code, "%s: %s" % (name, what))

        for what, kw in planar_faults(wmb):
            rc("in " + what, ARG, i=ok(pi, **kw))
            rc("base " + what, ARG, b=ok(pb, **kw))
            rc("out " + what, ARG, o=ok(po, **kw))
        rc("in with 2 channels", ARG, i=ok(pi, ch=2))
        rc("in with 3 channels", ARG, i=ok(pi, ch=3))
        rc("base with 4 channels", ARG, b=ok(pb, ch=4))
        rc("out with 4 channels", ARG, o=ok(po, ch=4))
        rc("base and out with 2 channels", ARG, b=ok(pb, ch=2), o=ok(po, ch=2))
        # two faults: the dims of a device image are compared first, those of a host image once it is staged
        first = DIMS if on_device else ARG
        rc("in: wrong dims and ld < cols", first, i=ok(pi, rows=ROWS + 1, ld=COLS - 1))
        rc("base: wrong dims and ld < cols", first, b=ok(pb, rows=ROWS + 1, ld=COLS - 1))
        rc("out: wrong dims and layout 99", first, o=ok(po, cols=COLS + 1, layout=99))
        rc("in: wrong dims, base: ld < cols", DIMS if on_device else ARG, i=ok(pi, rows=ROWS + 1), b=ok(pb, ld=COLS - 1))
        rc("in: ld < cols, base: wrong dims", ARG, i=ok(pi, ld=COLS - 1), b=ok(pb, rows=ROWS + 1))
        rc("in: wrong dims", DIMS, i=ok(pi, rows=ROWS + 1))
        rc("out: wrong dims", DIMS, o=ok(po, cols=COLS + 1))
        if name == "wm_embed_batch":  # batch strides of device batches are checked against one image
            one = ROWS * COLS
            rc("in stride < one image", ARG, s=(one - 1, 0, 0))
            rc("out stride < one image", ARG, s=(0, 0, one - 1))
            ps = one + 5  # three padded planes: one image spans 2 * ps + one elements
            rgb = lambda p: ok(p, ch=3, ps=ps)
            rc("RGB base stride < one image", ARG, b=rgb(pb), o=rgb(po), s=(0, 2 * ps + one - 1, 3 * ps))
            rc("RGB out stride < one image", ARG, b=rgb(pb), o=rgb(po), s=(0, 3 * ps, 2 * ps + one - 1))
            assert call(ok(pi), rgb(pb), rgb(po), (one, 2 * ps + one, 2 * ps + one)) == 0, "strides of exactly one image"
            assert wmb.lib().wm_sync(wm._h, 0) >= 0
        if name == "wm_embed_verify_host_batch":
            rc("out of another dtype", ARG, o=ok(po, dtype=wmb.U8))
            rc("RGB out", ARG, b=ok(pb, ch=3), o=ok(po, ch=3))


def test_detect_planar_faults(wmb, env):
    wm, dev, host = env
    for name, (on_device, call) in detect_forms(wmb, wm).items():
        p = dev[0] if on_device else host[0].ctypes.data

        def rc(what, code, s=0, **kw):
            expect(wmb, wm, call(desc(wmb, p, **kw), s), code, "%s: %s" % (name, what))

        for what, kw in planar_faults(wmb):
            rc(what, ARG, **kw)
        rc("2 channels", ARG, ch=2)
        rc("3 channels", ARG, ch=3)
        rc("wrong dims and ld < cols", DIMS if on_device else ARG, rows=ROWS + 1, ld=COLS - 1)
        rc("wrong dims and layout 99", DIMS if on_device else ARG, cols=COLS + 1, layout=99)
        rc("wrong dims", DIMS, rows=ROWS + 1)
        if name == "wm_detect_batch":
            rc("stride < one image", ARG, s=ROWS * COLS - 1)
            rc("col-major stride < one image", ARG, s=COLS * (ROWS + 3) - 1, layout=wmb.COL_MAJOR, ld=ROWS + 3)


def test_debug_entry_points(wmb, env):
    wm, dev, _ = env
    L = wmb.lib()
    corr = C.c_float(0)

    def plane(what, code, **kw):
        expect(wmb, wm, L.wm_debug_plane(wm._h, C.byref(desc(wmb, dev[0], **kw)), wmb.DBG_ERRSEQ, dev[2]), code, "wm_debug_plane: " + what)

    def planes(what, code, **kw):
        expect(wmb, wm, L.wm_debug_detect_planes(wm._h, C.byref(desc(wmb, dev[0], **kw)), wmb.ME, dev[1], dev[2], C.byref(corr)), code,
               "wm_debug_detect_planes: " + what)

    for what, kw in planar_faults(wmb):
        plane(what, ARG, **kw)
        planes(what, ARG, **kw)
    for ch in (2, 3):
        plane("%d channels" % ch, ARG, ch=ch)
        planes("%d channels" % ch, ARG, ch=ch)
    plane("wrong dims and ld < cols", DIMS, rows=ROWS + 1, ld=COLS - 1)
    plane("wrong dims", DIMS, cols=COLS + 1)
    plane("packed RGB", ARG, layout=wmb.PACKED_RGB, dtype=wmb.U8, ch=3)
    planes("packed RGB", ARG, layout=wmb.PACKED_RGB, dtype=wmb.U8, ch=3)
    planes("packed RGB with wrong dims", ARG, layout=wmb.PACKED_RGB, dtype=wmb.U8, ch=3, rows=ROWS + 1)
    planes("u8", ARG, dtype=wmb.U8)


# ---- the video driver ----
def video_code(wmb, wm, frames, height=ROWS, width=COLS, interval=1, linesize=0, layout=0, mode=None, has_out=True):
    v = wmb.VideoProcessingContext(wm, height, width, interval, linesize=linesize, layout=layout)
    scal = np.zeros(4, np.float32)
    mode = wmb.VIDEO_EMBED if mode is None else mode
    with pytest.raises(wmb.WatermarkError) as e:
        wmb.process_frames(v, mode, frames.ctypes.data, frames.ctypes.data + frames.nbytes // 2 if has_out else None, 0, 2, scal)
    print(e.value)
    return e.value.code


def test_video_frame_faults(wmb):
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    frames = np.zeros(4 * 2 * (ROWS + 1) * 4 * (COLS + 1), np.uint8)  # in and out of two frames of up to 4 bytes per pixel
    code = lambda **kw: video_code(wmb, wm, frames, **kw)
    for y in (0, wmb.ROW_MAJOR):  # Y planes
        assert code(layout=y, linesize=COLS - 1) == ARG
        assert code(layout=y, linesize=COLS - 1, mode=wmb.VIDEO_DETECT, has_out=False) == ARG
        assert code(layout=y, height=ROWS + 1) == DIMS
        assert code(layout=y, height=ROWS + 1, linesize=COLS - 1) == DIMS
        assert code(layout=y, width=COLS + 1, interval=0) == DIMS
        assert code(layout=y, height=ROWS + 1, mode=9) == ARG
        assert code(layout=y, linesize=COLS - 1, interval=0) == ARG
    for layout in (99, -1, 8):
        assert code(layout=layout) == ARG
        assert code(layout=layout, mode=wmb.VIDEO_DETECT, has_out=False) == ARG
        assert code(layout=layout, height=ROWS + 1) == DIMS
        assert code(layout=layout, has_out=False) == ARG
    assert code(layout=wmb.PACKED_BGR, linesize=3 * COLS - 1) == ARG
    assert code(layout=wmb.PACKED_BGRA, linesize=4 * COLS - 1, mode=wmb.VIDEO_EMBED_VERIFY) == ARG
    assert code(layout=wmb.PACKED_BGR, linesize=3 * COLS - 1, height=ROWS + 1) == DIMS
    assert code(layout=wmb.PACKED_UYVY, linesize=2 * COLS - 1, mode=wmb.VIDEO_DETECT, has_out=False) == ARG
    wm.close()
    wo = wmb.Watermark(ROWS, COLS + 1, util.normal_w(ROWS, COLS + 1), 3, PSNR)  # 4:2:2 frames have an even width
    assert video_code(wmb, wo, frames, width=COLS + 1, layout=wmb.PACKED_YUYV) == ARG
    assert video_code(wmb, wo, frames, width=COLS + 1, layout=wmb.PACKED_YUYV, height=ROWS + 1) == DIMS
    assert video_code(wmb, wo, frames, width=COLS + 1, layout=wmb.PACKED_UYVY, linesize=2 * COLS + 2) == ARG
    wo.close()


def run_y_frames(wmb, wm, buf, rows, cols, linesize, layout, mode, on_device):
    """wm_process_frames on the Y planes `buf` (n, rows, linesize), frames 1.. of the stream, interval 2 -> (out or None, scalars)"""
    n = buf.shape[0]
    embed = mode != wmb.VIDEO_DETECT
    scal = np.full(2 * n, 7.0, np.float32)
    if on_device:
        src = dev_raw(wmb, wm, buf)
        dst = dev_raw(wmb, wm, np.full(n * rows * cols, 0xA5, np.uint8)) if embed else None
    else:
        host_out = np.full(n * rows * cols, 0xA5, np.uint8)
        src, dst = buf.ctypes.data, host_out.ctypes.data if embed else None
    v = wmb.VideoProcessingContext(wm, rows, cols, 2, linesize=linesize, frames_on_device=on_device, layout=layout)
    assert wmb.process_frames(v, mode, src, dst, 1, n, scal) == n
    out = None
    if embed:
        out = dev_get(wmb, wm, dst, (n * rows * cols,)) if on_device else host_out
    if on_device:
        wmb.lib().wm_dev_free(wm._h, src)
        if dst:
            wmb.lib().wm_dev_free(wm._h, dst)
    return out, scal


@pytest.mark.parametrize("on_device", [False, True])
def test_video_layout_0_equals_row_major(wmb, on_device):
    rows, cols, n, linesize = 270, 480, 7, 512
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    buf = np.full((n, rows, linesize), 0x33, np.uint8)
    for i in range(n):
        buf[i, :, :cols] = util.natural_image(rows, cols, seed=i, integer=True)
    for mode in (wmb.VIDEO_EMBED_VERIFY, wmb.VIDEO_DETECT):
        o0, s0 = run_y_frames(wmb, wm, buf, rows, cols, linesize, 0, mode, on_device)
        o1, s1 = run_y_frames(wmb, wm, buf, rows, cols, linesize, wmb.ROW_MAJOR, mode, on_device)
        assert np.isfinite(s0).any(), mode
        assert np.array_equal(s0.view(np.uint32), s1.view(np.uint32)), mode
        if o0 is not None:
            assert np.array_equal(o0, o1), mode
    wm.close()
