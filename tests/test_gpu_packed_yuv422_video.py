"""Packed 4:2:2 frames (wm_video_ctx.layout = WM_PACKED_YUYV / UYVY) through the video driver.

A gated frame must get what the packed image entry points give it (wm_embed_batch / wm_detect_batch on that frame alone: bit for bit
when the driver also runs it alone, the correlation within 1e-6 relative when it shares a run with other frames).  Gated-off frames are
copied through without the row padding, both bytes of every pixel; the chroma is the input's on every frame.  On the same luma the driver
gives the luma bytes and `a` of the Y-plane driver, and its correlation within 1e-6 relative.
"""
import os
import subprocess

import numpy as np
import pytest

import util
from test_gpu_packed_rgb import dev_get, dev_raw
from test_gpu_packed_video import check, pitched, references, run_driver
from test_gpu_packed_yuv422 import chroma_plane, koff, luma_image, pack, round16

pytestmark = pytest.mark.gpu

PSNR = 40.0
ROWS, COLS = 540, 960


def layouts(wmb):
    return [wmb.PACKED_YUYV, wmb.PACKED_UYVY]


def make_frames(wmb, layout, rows, cols, n, seed=0):
    """n packed 4:2:2 frames (n, rows, cols, 2): natural lumas, seeded random chroma with 0 and 255"""
    ys = [luma_image(rows, cols, seed=seed + k) for k in range(3)]
    out = np.empty((n, rows, cols, 2), np.uint8)
    for i in range(n):
        out[i] = pack(wmb, np.roll(ys[i % 3], 11 * i, axis=1), chroma_plane(rows, cols, seed + i), layout)
    return out


def chroma_kept(wmb, out, frames, layout, what):
    k = koff(wmb, layout)
    assert np.array_equal(out[..., 1 - k], frames[..., 1 - k]), what


# ---- 1. runs of one frame: bit-identical to the single-image batch calls ----
@pytest.mark.parametrize("interval", [1, 3])
@pytest.mark.parametrize("on_device", [False, True])
@pytest.mark.parametrize("li", range(2))
def test_runs_of_one_frame(wmb, li, on_device, interval):
    layout = layouts(wmb)[li]
    n, first = 7, 4
    frames = make_frames(wmb, layout, ROWS, COLS, n, seed=li)
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    wm.set_option(wmb.OPT_HOST_RUN_FRAMES, 1)
    wm.set_option(wmb.OPT_RUN_MB, 1)  # a 540 x 960 4:2:2 frame is just under 1 MB: runs of one frame
    refs = references(wmb, wm, frames, layout, first, interval)
    out, a = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device, linesize=2 * COLS + 64)
    _, corr = run_driver(wmb, wm, out, layout, wmb.VIDEO_DETECT, interval, first, on_device)
    what = "layout=%d device=%d interval=%d" % (layout, on_device, interval)
    check(frames, first, interval, out, a, corr, refs, True, what)
    chroma_kept(wmb, out, frames, layout, what)
    wm.close()


# ---- 2. default run sizes, uneven runs ----
@pytest.mark.parametrize("interval", [1, 3])
@pytest.mark.parametrize("on_device", [False, True])
@pytest.mark.parametrize("li", range(2))
def test_default_runs(wmb, li, on_device, interval):
    """37 frames (host: runs of 4 and 3; device: runs of up to 32 frames, two of unequal length at interval 1)"""
    layout = layouts(wmb)[li]
    n, first = 37, 2
    frames = make_frames(wmb, layout, ROWS, COLS, n, seed=10 + li)
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    refs = references(wmb, wm, frames, layout, first, interval)
    out, a = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device)
    _, corr = run_driver(wmb, wm, out, layout, wmb.VIDEO_DETECT, interval, first, on_device)
    what = "layout=%d device=%d interval=%d" % (layout, on_device, interval)
    check(frames, first, interval, out, a, corr, refs, False, what)
    chroma_kept(wmb, out, frames, layout, what)
    wm.close()


# ---- 3. gated-off frames: both bytes copied through ----
@pytest.mark.parametrize("on_device", [False, True])
def test_gated_off_frames_copied(wmb, on_device):
    n, first, interval = 9, 1, 2
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    for layout in layouts(wmb):
        frames = make_frames(wmb, layout, ROWS, COLS, n, seed=20)
        for mode in (wmb.VIDEO_EMBED, wmb.VIDEO_EMBED_VERIFY):
            out, _ = run_driver(wmb, wm, frames, layout, mode, interval, first, on_device, linesize=2 * COLS + 64, fill=0xEE)
            gated = (first + np.arange(n)) % interval == 0
            assert np.array_equal(out[~gated], frames[~gated])
            chroma_kept(wmb, out, frames, layout, "layout=%d mode=%d" % (layout, mode))
            k = koff(wmb, layout)
            assert all(not np.array_equal(out[i, ..., k], frames[i, ..., k]) for i in np.nonzero(gated)[0])  # watermarked
    wm.close()


# ---- 4. EMBED_VERIFY = EMBED, then DETECT on that output ----
@pytest.mark.parametrize("on_device", [False, True])
def test_embed_verify_equals_embed_then_detect(wmb, on_device):
    n, first, interval = 11, 1, 2
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    for layout in layouts(wmb):
        frames = make_frames(wmb, layout, ROWS, COLS, n, seed=30)
        frames[3, ..., koff(wmb, layout)] = 117  # a constant luma at global index 4, gated on: unsolvable, `a` NaN, copied through, corr 0
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


# ---- 5. host row padding: padded linear upload, 2-D copy, WM_OPT_PADDED_UPLOAD = 0 ----
@pytest.mark.parametrize("li", range(2))
def test_host_row_padding(wmb, li):
    layout = layouts(wmb)[li]
    rowb = 2 * COLS
    n, first, interval = 10, 0, 1
    frames = make_frames(wmb, layout, ROWS, COLS, n, seed=50 + li)
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    ref_o, ref_s = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED_VERIFY, interval, first, False)
    for ls, padded_upload, fill in ((rowb + 64, 1, 0x00), (rowb + 64, 1, 0xFF), (rowb + 2, 1, 0xFF), (rowb + 64, 0, 0xFF)):
        wm.set_option(wmb.OPT_PADDED_UPLOAD, padded_upload)
        o, s = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED_VERIFY, interval, first, False, linesize=ls, fill=fill)
        what = "layout=%d linesize=%d padded_upload=%d fill=%d" % (layout, ls, padded_upload, fill)
        assert np.array_equal(o, ref_o), what
        assert np.array_equal(s.view(np.uint32), ref_s.view(np.uint32)), what
    wm.close()


# ---- 6. several contexts: contiguous chunks of the global frame index ----
@pytest.mark.parametrize("on_device", [False, True])
@pytest.mark.parametrize("nctx", [2, 3])
def test_multi_equals_single(wmb, nctx, on_device):
    n, first, interval = 23, 5, 3
    wm = wmb.Watermark(ROWS, COLS, util.normal_w(ROWS, COLS), 3, PSNR)
    clones = [wm.clone() for _ in range(nctx)]
    for layout in layouts(wmb):
        frames = make_frames(wmb, layout, ROWS, COLS, n, seed=60)
        ls = 2 * COLS + 64
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


# ---- 7. against the Y-plane driver on the same luma frames (device frames, linesize round_up(width, 16)) ----
def yplane_driver(wmb, wm, ys, mode, interval, first):
    """the Y-plane driver on device luma frames (n, rows, cols) at linesize round_up(cols, 16) -> (out (n, rows, cols), scalars)"""
    n, rows, cols = ys.shape
    ls = round16(cols)
    buf = np.zeros((n, rows, ls), np.uint8)
    buf[:, :, :cols] = ys
    src, dst = dev_raw(wmb, wm, buf), dev_raw(wmb, wm, np.zeros(n * rows * cols, np.uint8))
    scal = np.full(2 * n, 7.0, np.float32)
    v = wmb.VideoProcessingContext(wm, rows, cols, interval, linesize=ls, frames_on_device=True)
    assert wmb.process_frames(v, mode, src, dst, first, n, scal) == n
    out = dev_get(wmb, wm, dst, (n, rows, cols))
    for p in (src, dst):
        wmb.lib().wm_dev_free(wm._h, p)
    return out, scal


@pytest.mark.parametrize("rows,cols", [(540, 960), (540, 958)])
def test_equal_to_yplane_driver(wmb, rows, cols):
    n, first, interval = 19, 0, 1
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    for layout in layouts(wmb):
        frames = make_frames(wmb, layout, rows, cols, n, seed=80)
        k = koff(wmb, layout)
        ro, rs = yplane_driver(wmb, wm, np.ascontiguousarray(frames[..., k]), wmb.VIDEO_EMBED_VERIFY, interval, first)
        o, s = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED_VERIFY, interval, first, True)
        rc = float(np.max(np.abs(s[n:].astype(np.float64) - rs[n:]) / np.abs(rs[n:])))
        print("vs Y-plane driver %dx%d layout=%d: differing luma bytes %d, corr max rel %.3g" % (
            rows, cols, layout, int(np.count_nonzero(o[..., k] != ro)), rc))
        assert np.array_equal(o[..., k], ro)
        assert np.array_equal(o[..., 1 - k], frames[..., 1 - k])
        assert np.array_equal(s[:n].view(np.uint32), rs[:n].view(np.uint32))
        assert rc <= 1e-6
    wm.close()


# ---- 8. against the CPU oracle ----
def test_against_oracle(wmb, oracle):
    rows, cols = 1080, 1920
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    for layout, on_device in ((wmb.PACKED_YUYV, False), (wmb.PACKED_UYVY, True)):
        frames = make_frames(wmb, layout, rows, cols, 1, seed=40)
        k = koff(wmb, layout)
        out, s = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED_VERIFY, 1, 0, on_device)
        est, eo, ea = oracle.embed_frame_u8(frames[0, ..., k], W, PSNR, oracle.ME)
        dst, dcorr = oracle.detect_frame_u8(eo, W, oracle.ME)
        dpx = np.abs(out[0, ..., k].astype(int) - eo.astype(int)).max()
        ra, rc = util.rel(s[0], ea), util.rel(s[1], dcorr)
        print("oracle layout=%d: a rel %.3g corr rel %.3g max luma diff %d" % (layout, ra, rc, dpx))
        assert est == 0 and dst == 0 and ra <= 1e-3 and rc <= 1e-3 and dpx <= 1
        assert np.array_equal(out[0, ..., 1 - k], frames[0, ..., 1 - k])
    wm.close()


# ---- 9. rejections ----
def test_rejections(wmb):
    rows, n = 67, 2
    frames = np.zeros((n, rows, 4 * 131), np.uint8)
    out = np.zeros_like(frames)
    scal = np.zeros(2 * n, np.float32)

    def refused(wm, cols, layout, linesize, mode, has_out, what):
        v = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=linesize, layout=layout)
        with pytest.raises(wmb.WatermarkError) as e:
            wmb.process_frames(v, mode, frames.ctypes.data, out.ctypes.data if has_out else None, 0, n, scal)
        print("%s: %s" % (what, e.value))
        assert e.value.code == -5, what

    even = wmb.Watermark(rows, 130, util.normal_w(rows, 130), 3, PSNR)
    odd = wmb.Watermark(rows, 131, util.normal_w(rows, 131), 3, PSNR)
    refused(even, 130, wmb.PACKED_YUYV, 2 * 130 - 1, wmb.VIDEO_EMBED, True, "YUYV linesize < 2 * width")
    refused(even, 130, wmb.PACKED_UYVY, 2 * 130 - 1, wmb.VIDEO_DETECT, False, "UYVY linesize < 2 * width")
    refused(odd, 131, wmb.PACKED_YUYV, 0, wmb.VIDEO_EMBED, True, "YUYV odd width")
    refused(odd, 131, wmb.PACKED_UYVY, 4 * 131, wmb.VIDEO_DETECT, False, "UYVY odd width")
    refused(even, 130, wmb.PACKED_YUYV, 0, wmb.VIDEO_EMBED, False, "embed without out")
    for layout in (8, 9):
        refused(even, 130, layout, 4 * 130, wmb.VIDEO_EMBED, True, "layout %d" % layout)
    assert np.all(out == 0)
    even.close()
    odd.close()


# ---- 10. the C++ façade: processFramesInMemory on YUYV frames, one and two Watermark objects ----
def test_cpp_process_frames_in_memory_yuyv(wmb, tmp_path):
    b = wmb.build()
    exe = b.build_video_yuv422_test()
    assert exe and os.path.exists(exe)
    rows, cols, n, interval = 120, 200, 7, 2
    ls = 2 * cols + 24
    W = util.normal_w(rows, cols)
    frames = make_frames(wmb, wmb.PACKED_YUYV, rows, cols, n, seed=70)
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
    out, a = run_driver(wmb, wm, frames, wmb.PACKED_YUYV, wmb.VIDEO_EMBED, interval, 0, False, linesize=ls)
    _, corr = run_driver(wmb, wm, out, wmb.PACKED_YUYV, wmb.VIDEO_DETECT, interval, 0, False)
    assert np.array_equal(np.fromfile(tmp_path / "out.u8", np.uint8).reshape(out.shape), out)
    for i in range(n):
        assert np.array_equal(np.float32(got["a_%d" % i]), a[i], equal_nan=True)
        assert np.array_equal(np.float32(got["corr_%d" % i]), corr[i], equal_nan=True)
    wm.close()
