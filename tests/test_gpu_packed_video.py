"""Packed colour frames (wm_video_ctx.layout = WM_PACKED_RGB / BGR / RGBA / BGRA) through the video driver.

A gated frame must get what the packed image entry points give it: the output bytes, `a` and the correlation of wm_embed_batch /
wm_detect_batch run on that frame alone (bit for bit when the driver also runs it alone; the correlation within 1e-6 relative when it
shares a run with other frames, as for packed batches in test_gpu_packed_rgb.py::test_batches).  Gated-off frames are copied through
without the row padding, every byte of a pixel; the fourth byte of a 4-byte frame is the input's on every frame.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import util
from test_gpu_packed_rgb import color_image, dev_get, dev_raw, f32bits

pytestmark = pytest.mark.gpu

PSNR = 40.0
ROWS, COLS = 540, 960  # a BGR frame is 1.5 MB: WM_OPT_RUN_MB = 1 gives runs of one frame


def layouts(wmb):
    return [wmb.PACKED_RGB, wmb.PACKED_BGR, wmb.PACKED_RGBA, wmb.PACKED_BGRA]


def make_frames(wmb, layout, rows, cols, n, seed=0):
    """n packed frames (n, rows, cols, bpp): colour images, B and R swapped for the BGR orders, seeded alpha for the 4-byte layouts"""
    bpp = wmb.PACKED_BYTES[layout]
    base = [color_image(rows, cols, seed=seed + k) for k in range(3)]
    rng = np.random.default_rng(500 + seed)
    out = np.empty((n, rows, cols, bpp), np.uint8)
    for i in range(n):
        img = np.roll(base[i % 3], 11 * i, axis=1)
        out[i, ..., :3] = img[..., ::-1] if layout in (wmb.PACKED_BGR, wmb.PACKED_BGRA) else img
        if bpp == 4:
            alpha = rng.integers(0, 256, (rows, cols), dtype=np.uint8)
            alpha[0, 0], alpha[-1, -1] = 0, 255
            out[i, ..., 3] = alpha
    return out


def pitched(frames, linesize, fill):
    """frames (n, rows, cols, bpp) -> (n, rows, linesize) bytes, the row padding set to `fill`"""
    n, rows, cols, bpp = frames.shape
    buf = np.full((n, rows, linesize), fill, np.uint8)
    buf[:, :, :bpp * cols] = frames.reshape(n, rows, bpp * cols)
    return buf


def run_driver(wmb, wm, frames, layout, mode, interval, first, on_device, linesize=0, fill=0x33, ctxs=None):
    """wm_process_frames (or wm_process_frames_multi over the contexts `ctxs`) on `frames` -> (out (n, rows, cols, bpp) or None, scalars)"""
    n, rows, cols, bpp = frames.shape
    ls = linesize or bpp * cols
    buf = pitched(frames, ls, fill)
    obytes = rows * bpp * cols
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
        v = wmb.VideoProcessingContext(wm, rows, cols, interval, linesize=linesize, frames_on_device=on_device, layout=layout)
        assert wmb.process_frames(v, mode, src, dst, first, n, scal) == n
    else:
        vs = [wmb.VideoProcessingContext(c, rows, cols, interval, linesize=linesize, frames_on_device=on_device, layout=layout) for c in ctxs]
        firsts = [wmb.shard_frames(n, g, len(ctxs))[0] for g in range(len(ctxs))]
        got = wmb.process_frames_multi(vs, mode, [src + f * rows * ls for f in firsts], [dst + f * obytes for f in firsts] if embed else None,
                                       first, n, scal)
        assert got == n
    out = None
    if embed:
        out = dev_get(wmb, wm, dst, (n, obytes)) if on_device else host_out
        out = out.reshape(n, rows, cols, bpp)
    if on_device:
        L.wm_dev_free(wm._h, src)
        if embed:
            L.wm_dev_free(wm._h, dst)
    return out, scal


def per_frame(wmb, wm, frame, layout):
    """wm_embed_batch + wm_detect_batch with batch 1 on one dense frame -> (out, a, corr) as the video driver reports them"""
    rows, cols, bpp = frame.shape
    pin, pout = dev_raw(wmb, wm, frame), dev_raw(wmb, wm, np.zeros_like(frame))
    desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, 0, bpp)
    a, st, corr, st2 = np.full(1, np.nan, np.float32), np.zeros(1, np.int32), np.zeros(1, np.float32), np.zeros(1, np.int32)
    wm.embed_batch(0, desc(pin), desc(pin), desc(pout), 0, 0, 0, 1, wmb.ME, a, st)
    wm.detect_batch(0, desc(pout), 0, 1, wmb.ME, corr, st2)
    wm.sync(0)
    out = dev_get(wmb, wm, pout, frame.shape)
    for p in (pin, pout):
        wmb.lib().wm_dev_free(wm._h, p)
    # the driver leaves `a` NaN for an unsolvable frame and reports its correlation as 0 (Watermark.cpp:164-165,246-247)
    return out, (np.float32(np.nan) if st[0] == wmb.SINGULAR else a[0]), (corr[0] if st2[0] == 0 else np.float32(0))


def check(frames, first, interval, out, a, corr, refs, exact_corr, what):
    """out / a / corr of a driver run against the per-frame references of the gated frames"""
    n = frames.shape[0]
    gated = (first + np.arange(n)) % interval == 0
    assert np.all(np.isnan(a[~gated])) and np.all(np.isnan(corr[~gated])), what
    for i in range(n):
        if out is not None:
            if frames.shape[3] == 4:
                assert np.array_equal(out[i, ..., 3], frames[i, ..., 3]), (what, i)  # the fourth byte, gated or not
            if not gated[i]:
                assert np.array_equal(out[i], frames[i]), (what, i)
        if gated[i]:
            ro, ra, rc = refs[i]
            if out is not None:
                assert np.array_equal(out[i], ro), (what, i, int(np.count_nonzero(out[i] != ro)))
            assert (np.isnan(a[i]) and np.isnan(ra)) or f32bits(a[i]) == f32bits(ra), (what, i, a[i], ra)
            if exact_corr:
                assert f32bits(corr[i]) == f32bits(rc), (what, i, corr[i], rc)
            else:
                assert abs(float(corr[i]) - float(rc)) <= 1e-6 * abs(float(rc)), (what, i, corr[i], rc)


def references(wmb, wm, frames, layout, first, interval):
    return {i: per_frame(wmb, wm, frames[i], layout) for i in range(frames.shape[0]) if (first + i) % interval == 0}


# ---- 1. runs of one frame: bit-identical to the single-image batch calls ----
@pytest.mark.parametrize("interval", [1, 3])
@pytest.mark.parametrize("on_device", [False, True])
@pytest.mark.parametrize("li", range(4))
def test_runs_of_one_frame(wmb, li, on_device, interval):
    layout = layouts(wmb)[li]
    n, first = 7, 4
    frames = make_frames(wmb, layout, ROWS, COLS, n, seed=li)
    assert frames[0].nbytes > 2**20
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    wm.set_option(wmb.OPT_HOST_RUN_FRAMES, 1)
    wm.set_option(wmb.OPT_RUN_MB, 1)
    refs = references(wmb, wm, frames, layout, first, interval)
    ls = wmb.PACKED_BYTES[layout] * COLS + 64
    out, a = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device, linesize=ls)
    _, corr = run_driver(wmb, wm, out, layout, wmb.VIDEO_DETECT, interval, first, on_device)
    check(frames, first, interval, out, a, corr, refs, True, "layout=%d device=%d interval=%d" % (layout, on_device, interval))
    wm.close()


# ---- 2. default run sizes, uneven runs ----
@pytest.mark.parametrize("interval", [1, 3])
@pytest.mark.parametrize("on_device", [False, True])
@pytest.mark.parametrize("li", range(4))
def test_default_runs(wmb, li, on_device, interval):
    """37 frames (host: runs of 4 and 3; device: runs of up to 32 frames, two of unequal length at interval 1)"""
    layout = layouts(wmb)[li]
    n, first = 37, 2
    frames = make_frames(wmb, layout, ROWS, COLS, n, seed=10 + li)
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    refs = references(wmb, wm, frames, layout, first, interval)
    out, a = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device)
    _, corr = run_driver(wmb, wm, out, layout, wmb.VIDEO_DETECT, interval, first, on_device)
    check(frames, first, interval, out, a, corr, refs, False, "layout=%d device=%d interval=%d" % (layout, on_device, interval))
    wm.close()


# ---- 3. the fourth byte ----
@pytest.mark.parametrize("on_device", [False, True])
def test_fourth_byte_copied_on_every_frame(wmb, on_device):
    n = 9
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    for layout in (wmb.PACKED_RGBA, wmb.PACKED_BGRA):
        frames = make_frames(wmb, layout, ROWS, COLS, n, seed=20)
        for mode in (wmb.VIDEO_EMBED, wmb.VIDEO_EMBED_VERIFY):
            out, _ = run_driver(wmb, wm, frames, layout, mode, 2, 1, on_device, linesize=4 * COLS + 64)
            assert np.array_equal(out[..., 3], frames[..., 3])
            assert not np.array_equal(out[1, ..., :3], frames[1, ..., :3])  # frame 1 (global index 2) is gated on: watermarked
    wm.close()


# ---- 4. EMBED_VERIFY = EMBED, then DETECT on that output ----
@pytest.mark.parametrize("on_device", [False, True])
def test_embed_verify_equals_embed_then_detect(wmb, on_device):
    n, first, interval = 11, 1, 2
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    for layout in layouts(wmb):
        frames = make_frames(wmb, layout, ROWS, COLS, n, seed=30)
        frames[3, ..., :3] = (10, 200, 31)  # a constant frame at global index 4, gated on: unsolvable, `a` NaN, copied through, correlation 0
        ov, sv = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED_VERIFY, interval, first, on_device)
        oe, a = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device)
        _, corr = run_driver(wmb, wm, oe, layout, wmb.VIDEO_DETECT, interval, first, on_device)
        assert np.array_equal(ov, oe)
        assert np.array_equal(sv[:n].view(np.uint32), a.view(np.uint32))
        assert np.array_equal(sv[n:].view(np.uint32), corr.view(np.uint32))
        assert np.isnan(a[3]) and corr[3] == 0.0 and np.array_equal(ov[3], frames[3])
        gated = (first + np.arange(n)) % interval == 0
        assert not np.any(np.isnan(a[gated & (np.arange(n) != 3)]))
    wm.close()


# ---- 5. against the CPU oracle ----
@pytest.mark.parametrize("which", ["1080p_bgr_host", "4k_bgra_device"])
def test_against_oracle(wmb, oracle, which):
    rows, cols, layout, on_device = (1080, 1920, wmb.PACKED_BGR, False) if which.startswith("1080p") else (2160, 3840, wmb.PACKED_BGRA, True)
    frames = make_frames(wmb, layout, rows, cols, 1, seed=40)
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    out, s = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED_VERIFY, 1, 0, on_device)
    rgb = np.ascontiguousarray(frames[0, ..., 2::-1].transpose(2, 0, 1)).astype(np.float32)  # B,G,R(,A) -> planar R,G,B
    e = oracle.embed(oracle.rgb2gray(rgb), W, PSNR, oracle.ME, base=rgb)
    trunc = e["out"].astype(np.uint8)
    corr_ref = oracle.detect(oracle.rgb2gray(trunc.astype(np.float32)), W, oracle.ME)["corr"]
    dpx = np.abs(out[0, ..., 2::-1].astype(int) - trunc.transpose(1, 2, 0).astype(int)).max()
    ra, rc = util.rel(s[0], e["a"]), util.rel(s[1], corr_ref)
    print("oracle %s: a rel %.3g corr rel %.3g max pixel diff %d" % (which, ra, rc, dpx))
    assert e["status"] == 0 and ra <= 1e-3 and rc <= 1e-3 and dpx <= 1
    if layout == wmb.PACKED_BGRA:
        assert np.array_equal(out[0, ..., 3], frames[0, ..., 3])
    wm.close()


# ---- 6. host row padding: padded linear upload, 2-D copy, WM_OPT_PADDED_UPLOAD = 0 ----
@pytest.mark.parametrize("li", range(4))
def test_host_row_padding(wmb, li):
    layout = layouts(wmb)[li]
    rowb = wmb.PACKED_BYTES[layout] * COLS
    n, first, interval = 10, 0, 1
    frames = make_frames(wmb, layout, ROWS, COLS, n, seed=50 + li)
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    ref_o, ref_s = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED_VERIFY, interval, first, False)
    for ls, padded_upload, fill in ((rowb + 64, 1, 0x00), (rowb + 64, 1, 0xFF), (rowb + 5, 1, 0xFF), (rowb + 64, 0, 0xFF)):
        wm.set_option(wmb.OPT_PADDED_UPLOAD, padded_upload)
        o, s = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED_VERIFY, interval, first, False, linesize=ls, fill=fill)
        what = "layout=%d linesize=%d padded_upload=%d fill=%d" % (layout, ls, padded_upload, fill)
        assert np.array_equal(o, ref_o), what
        assert np.array_equal(s.view(np.uint32), ref_s.view(np.uint32)), what
    wm.close()


# ---- 7. several contexts: contiguous chunks of the global frame index ----
@pytest.mark.parametrize("on_device", [False, True])
@pytest.mark.parametrize("nctx", [2, 3])
def test_multi_equals_single(wmb, nctx, on_device):
    n, first, interval = 23, 5, 3
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    clones = [wm.clone() for _ in range(nctx)]
    for layout in (wmb.PACKED_BGR, wmb.PACKED_RGBA):
        frames = make_frames(wmb, layout, ROWS, COLS, n, seed=60)
        ls = wmb.PACKED_BYTES[layout] * COLS + 64
        o1, a1 = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device, linesize=ls)
        o2, a2 = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device, linesize=ls, ctxs=clones)
        assert np.array_equal(o1, o2)
        assert np.array_equal(a1.view(np.uint32), a2.view(np.uint32))
        _, c1 = run_driver(wmb, wm, o1, layout, wmb.VIDEO_DETECT, interval, first, on_device)
        _, c2 = run_driver(wmb, wm, o1, layout, wmb.VIDEO_DETECT, interval, first, on_device, ctxs=clones)
        gated = (first + np.arange(n)) % interval == 0
        assert np.all(np.isnan(c2[~gated])) and not np.any(np.isnan(c2[gated]))
        assert np.max(np.abs(c1[gated].astype(np.float64) - c2[gated]) / np.abs(c1[gated])) <= 1e-6
    for c in clones:
        c.close()
    wm.close()


# ---- 8. rejections ----
def test_rejections(wmb):
    rows, cols, n = 67, 131, 2
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    frames = np.zeros((n, rows, 4 * cols), np.uint8)
    out = np.zeros_like(frames)
    scal = np.zeros(2 * n, np.float32)

    def refused(layout, linesize, mode, has_out, what):
        v = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=linesize, layout=layout)
        with pytest.raises(wmb.WatermarkError) as e:
            wmb.process_frames(v, mode, frames.ctypes.data, out.ctypes.data if has_out else None, 0, n, scal)
        print("%s: %s" % (what, e.value))
        assert e.value.code == -5, what

    refused(6, 4 * cols, wmb.VIDEO_EMBED, True, "layout 6")
    refused(-1, 4 * cols, wmb.VIDEO_DETECT, False, "layout -1")
    refused(wmb.PACKED_BGR, 3 * cols - 1, wmb.VIDEO_EMBED, True, "BGR linesize < 3 * width")
    refused(wmb.PACKED_RGBA, 4 * cols - 1, wmb.VIDEO_DETECT, False, "RGBA linesize < 4 * width")
    refused(wmb.PACKED_BGRA, 0, wmb.VIDEO_EMBED, False, "embed without out")
    refused(wmb.PACKED_RGB, 0, wmb.VIDEO_EMBED_VERIFY, False, "embed + verify without out")
    wm.close()


# ---- 9. the C++ façade: processFramesInMemory on packed BGR frames, one and two Watermark objects ----
def test_cpp_process_frames_in_memory_bgr(wmb, tmp_path):
    b = wmb.build()
    exe = b.build_video_packed_test()
    assert exe and os.path.exists(exe)
    rows, cols, n, interval = 120, 200, 7, 2
    ls = 3 * cols + 24
    W = util.normal_w(rows, cols)
    frames = make_frames(wmb, wmb.PACKED_BGR, rows, cols, n, seed=70)
    pitched(frames, ls, 0x77).tofile(tmp_path / "frames.u8")
    W.tofile(tmp_path / "w.dat")
    r = subprocess.run([exe, str(tmp_path / "w.dat"), str(rows), str(cols), str(tmp_path / "frames.u8"), str(n), str(ls), str(interval),
                        str(tmp_path / "out.u8")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = dict(line.split(None, 1) for line in r.stdout.strip().splitlines())
    assert got["frames"].split() == [str(n), str(n)]
    assert got["equal_pixels"].strip() == "1" and got["equal_a"].strip() == "1" and got["nan_where_gated_off"].strip() == "1"
    assert float(got["corr_max_rel"]) <= 1e-6
    # the façade's one-object run is the Python driver's run
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    out, a = run_driver(wmb, wm, frames, wmb.PACKED_BGR, wmb.VIDEO_EMBED, interval, 0, False, linesize=ls)
    _, corr = run_driver(wmb, wm, out, wmb.PACKED_BGR, wmb.VIDEO_DETECT, interval, 0, False)
    assert np.array_equal(np.fromfile(tmp_path / "out.u8", np.uint8).reshape(out.shape), out)
    for i in range(n):
        assert np.array_equal(np.float32(got["a_%d" % i]), a[i], equal_nan=True)
        assert np.array_equal(np.float32(got["corr_%d" % i]), corr[i], equal_nan=True)
    wm.close()
