"""The 8-bit kernels one by one at full frame sizes, each against a reference of its own operation built from the GPU's own inputs to
that kernel (u8_exact.py): the Rx sweep and the mask planes bit for bit, the stats kernel's sum2 and `a` within their derived bounds,
the apply kernel's bytes with no difference allowed, the detector's three sums and its correlation within their derived bounds.  Every
path that runs these kernels on u8 frames is checked on its own: the video driver on device and on host frames, the batch API with
both masks and p in {3, 5}, the replayed synchronous calls, and each option that must not change the bits."""
import ctypes as C
import functools

import numpy as np
import pytest

import u8_exact as X
import util
from test_gpu_parity import report

pytestmark = pytest.mark.gpu

SIZE_IDS = ["%dx%d_ls%d" % s for s in X.SIZES]
FULL_4K = (2160, 3840)


def _check(what, observed, bound):
    ratio = observed / bound
    report("u8 full size %s: observed %.3g bound %.3g ratio %.3f" % (what, observed, bound, ratio))
    assert observed <= bound, (what, observed, bound)


def _k(opts, ld, cols, bstride=None):
    return X.chain_len(128 if X.narrow_u8(opts, ld, cols, bstride) else 256)


def _wm(wmb, rows, cols, W, p=3, opts=None):
    wm = wmb.Watermark(rows, cols, W, p, 40.0)
    for name, v in (opts or {}).items():
        wm.set_option(getattr(wmb, "OPT_" + name), v)
    return wm


def _input_planes(wmb, wm, img, mask):
    """The GPU's own planes of a frame the stats and apply kernels read: (e = I - pred or None, mask plane)."""
    d = wmb.DeviceArray.from_numpy(wm, img, wmb.ROW_MAJOR)
    if mask == wmb.ME:
        e, m = wm.debug_plane(d, wmb.DBG_ERRSEQ), wm.debug_plane(d, wmb.DBG_MASK_ME)
    else:
        e, m = None, wm.debug_plane(d, wmb.DBG_MASK_NVF)
    d.free()
    return e, m


def check_stats(what, k, sf, W, e, m, a, sum2=None, emax=None):
    """Check 3: `a` (and the stats kernel's sum2 and max|e| where the call exposes them) against f64 sums over the GPU's own planes.
    ME: the kernel sums (|e| W)^2 and divides the norm by max|e| afterwards; NVF: (mask W)^2."""
    n = W.size
    x = (np.abs(e) if e is not None else m).astype(np.float32) * W
    s_ref = float(np.sum(np.square(x.astype(np.float64))))
    nrm = np.sqrt(s_ref)
    if e is not None:
        mx = np.float32(np.abs(e).max())
        if emax is not None:
            assert emax == mx, (what, emax, mx)
        nrm = nrm / float(mx)
    a_ref = sf / (nrm / np.sqrt(float(n)))
    if sum2 is not None:
        _check("%s sum2 k=%d" % (what, k), abs(sum2 - s_ref), X.sum_rel_bound(k, n) * s_ref)
    _check("%s a k=%d" % (what, k), abs(a - a_ref), X.a_rel_bound(k, n) * a_ref)


def check_apply(what, oracle, img, m, W, a, got, got_f32=None):
    """Check 4: the output bytes are those of the oracle's apply step on the GPU's mask plane and `a`, with no difference allowed."""
    v, want = X.apply_ref(oracle, img, m, W, a)
    lo, hi = X.clamps_fired(img, m, W, a)
    bad = X.unequal_bytes(got, want)
    report("u8 full size %s apply: unequal bytes %d of %d (clamped at 0: %d, at 255: %d)" % (what, bad, img.size, lo, hi))
    assert lo > 0 and hi > 0, (what, lo, hi)
    assert bad == 0, (what, bad, np.argwhere(got != want)[:5].tolist())
    if got_f32 is not None:
        badf = int(np.count_nonzero(got_f32.view(np.uint32) != v.view(np.uint32)))
        report("u8 full size %s apply f32 output: unequal values %d" % (what, badf))
        assert badf == 0, what


def _sums(ez, eu):
    ez, eu = ez.astype(np.float64), eu.astype(np.float64)
    return float(np.dot(eu.ravel(), ez.ravel())), float(np.dot(ez.ravel(), ez.ravel())), float(np.dot(eu.ravel(), eu.ravel()))


def check_detect(what, wmb, wm, oracle, z, W, mask, k, corr, sums=None, p=3):
    """Check 5: the detector's sums (where the call exposes them) and its correlation against f64 sums of the planes of the watermarked
    frame z.  p = 3: the GPU's own planes (DBG_ERRSEQ and the detector kernel's u, e_u on an f32 copy of z; that kernel's own sums are
    checked too, with the chain of the f32 detector).  p = 5: the NVF planes come from the oracle (the plane-writing detector takes 3 x 3
    masks only), so only the correlation is checked."""
    n = W.size
    if mask == wmb.NVF and p != 3:
        od = oracle.detect(z.astype(np.float32), W, wmb.NVF, o=oracle.opts(p=p))
        assert od["status"] == 0
        dot, nz, nu = _sums(od["ez"], od["eu"])
    else:
        dz = wmb.DeviceArray.from_numpy(wm, z.astype(np.float32), wmb.ROW_MAJOR)
        u, eu, corr32 = wm.debug_detect_planes(dz, mask)
        s32 = wm.debug(wmb.DBG_SCALARS)
        ez = wm.debug_plane(dz, wmb.DBG_ERRSEQ)
        dz.free()
        if mask == wmb.ME:  # the kernel keeps |e_z| W: the 1 / max|e| scale cancels in the correlation
            assert np.array_equal(u, np.abs(ez) * W), what
        dot, nz, nu = _sums(ez, eu)
        k32 = X.chain_len(256)
        _check("%s detector f32 dot k=%d" % (what, k32), abs(s32[4] - dot), X.dot_abs_bound(k32, n, nz, nu))
        _check("%s detector f32 nz k=%d" % (what, k32), abs(s32[5] - nz), X.sum_rel_bound(k32, n) * nz)
        _check("%s detector f32 nu k=%d" % (what, k32), abs(s32[6] - nu), X.sum_rel_bound(k32, n) * nu)
    if sums is not None:
        _check("%s dot k=%d" % (what, k), abs(sums[0] - dot), X.dot_abs_bound(k, n, nz, nu))
        _check("%s nz k=%d" % (what, k), abs(sums[1] - nz), X.sum_rel_bound(k, n) * nz)
        _check("%s nu k=%d" % (what, k), abs(sums[2] - nu), X.sum_rel_bound(k, n) * nu)
    _check("%s corr k=%d" % (what, k), abs(corr - dot / np.sqrt(nz * nu)), X.corr_abs_bound(k, n, dot, nz, nu))


@functools.lru_cache(maxsize=None)
def _frame(rows, cols, seed):
    return X.frame(rows, cols, seed)


@functools.lru_cache(maxsize=None)
def _w(rows, cols):
    return util.normal_w(rows, cols)


def _padded(img, ls):
    buf = np.full((img.shape[0], ls), 77, np.uint8)  # row padding holds bytes that must never be read as pixels
    buf[:, :img.shape[1]] = img
    return buf


# ---------------------------------------------------------------------------------------------------
# checks 1 and 2: the Rx sweep, the solve and the planes, bit for bit at full size
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,cols,ls", X.SIZES, ids=SIZE_IDS)
def test_sweep_and_planes_bit_exact(wmb, oracle, rows, cols, ls):
    img = _frame(rows, cols, 31)
    W = _w(rows, cols)
    f = img.astype(np.float32)
    wm = _wm(wmb, rows, cols, W)
    d = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.U8, 1, ls)
    d.upload(img)
    wm.detectWatermark(d, wmb.ME)
    Rx, rx, coef = wm.debug(wmb.DBG_RX), wm.debug(wmb.DBG_RXVEC), wm.debug(wmb.DBG_COEFFS)
    oRx, orx = oracle.rx(f)
    st, oc = oracle.solve8(Rx, rx)
    assert np.array_equal(Rx, oRx) and np.array_equal(rx, orx)
    assert st == 0 and np.array_equal(coef, oc.astype(np.float32))
    pe = oracle.pred_error_mask(f)
    planes = {"errseq": (wm.debug_plane(d, wmb.DBG_ERRSEQ), pe["e"]), "mask_me": (wm.debug_plane(d, wmb.DBG_MASK_ME), pe["mask"]),
              "mask_nvf": (wm.debug_plane(d, wmb.DBG_MASK_NVF), oracle.nvf(f))}
    wm.close()
    wm5 = _wm(wmb, rows, cols, W, p=5)
    d5 = wmb.DeviceArray(wm5, rows, cols, wmb.ROW_MAJOR, wmb.U8, 1, ls)
    d5.upload(img)
    planes["mask_nvf_p5"] = (wm5.debug_plane(d5, wmb.DBG_MASK_NVF), oracle.nvf(f, oracle.opts(p=5)))
    wm5.close()
    for name, (got, want) in planes.items():
        bad = int(np.count_nonzero(got.view(np.uint32) != want.view(np.uint32)))
        report("u8 full size %dx%d ls=%d plane %s: unequal values %d" % (rows, cols, ls, name, bad))
        assert bad == 0, name


# ---------------------------------------------------------------------------------------------------
# checks 3-5 on the synchronous calls (the third call of each is a graph replay), default options and each option that must not
# change the bits set away from its default
# ---------------------------------------------------------------------------------------------------
def _sync_checks(wmb, oracle, rows, cols, ls, mask, opts, tag):
    img = _frame(rows, cols, 47)
    W = _w(rows, cols)
    wm = _wm(wmb, rows, cols, W, opts=opts)
    sf = wm.strength_factor
    d = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.U8, 1, ls)
    d.upload(img)
    out = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.U8)
    out32 = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.F32)
    for _ in range(3):
        _, a, st = wm.makeWatermark(d, d, mask, out=out)
    assert st == 0
    s = wm.debug(wmb.DBG_SCALARS)
    assert s[1] == np.float32(a)
    for _ in range(3):
        _, a32, st = wm.makeWatermark(d, d, mask, out=out32)
    assert st == 0 and a32 == a
    z, z32 = out.numpy(), out32.numpy()
    for _ in range(3):
        corr, st = wm.detectWatermark(out, mask)
    assert st == 0
    sd = wm.debug(wmb.DBG_SCALARS)
    what = "%s %dx%d ls=%d mask=%d sync" % (tag, rows, cols, ls, mask)
    e, m = _input_planes(wmb, wm, img, mask)
    check_stats(what, _k(opts, ls, cols), sf, W, e, m, a, sum2=s[3], emax=s[2] if mask == wmb.ME else None)
    check_apply(what, oracle, img, m, W, a, z, z32)
    check_detect(what, wmb, wm, oracle, z, W, mask, _k(opts, cols, cols), corr, sums=sd[4:7])
    wm.close()


@pytest.mark.parametrize("mask", [0, 1])
@pytest.mark.parametrize("rows,cols,ls", X.SIZES, ids=SIZE_IDS)
def test_sync_calls(wmb, oracle, rows, cols, ls, mask):
    _sync_checks(wmb, oracle, rows, cols, ls, mask, {}, "defaults")


SAME_BITS_OPTIONS = [("NARROW_U8", 0), ("USE_TMA", 0), ("TMA_STORE", 0), ("PDL", 0), ("MMA_ACCUM", 0)]


@pytest.mark.parametrize("opt,value", SAME_BITS_OPTIONS, ids=[o for o, _ in SAME_BITS_OPTIONS])
@pytest.mark.parametrize("rows,cols,ls", [(1080, 1920, 1920), (130, 264, 272)], ids=["1080x1920", "130x264_ls272"])
def test_same_bits_options_each_meet_the_checks(wmb, oracle, rows, cols, ls, opt, value):
    for mask in (wmb.ME, wmb.NVF):
        _sync_checks(wmb, oracle, rows, cols, ls, mask, {opt: value}, "%s=%d" % (opt, value))


# ---------------------------------------------------------------------------------------------------
# checks 3-5 on the batch API: u8 images with both masks, the 3 x 3 NVF mask fused into the kernels (p = 3) and the precomputed mask
# planes of a 5 x 5 window (p = 5)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p", [3, 5])
@pytest.mark.parametrize("rows,cols,ls", X.SIZES, ids=SIZE_IDS)
def test_batch_calls(wmb, oracle, rows, cols, ls, p):
    B = 2
    W = _w(rows, cols)
    imgs = [_frame(rows, cols, 61 + b) for b in range(B)]
    wm = _wm(wmb, rows, cols, W, p=p)
    sf = wm.strength_factor
    L = wmb.lib()
    src = np.ascontiguousarray(np.stack([_padded(i, ls) for i in imgs]))
    din = L.wm_dev_alloc(wm._h, src.nbytes)
    dout = L.wm_dev_alloc(wm._h, B * rows * cols)
    L.wm_dev_upload(wm._h, din, src.ctypes.data, src.nbytes)
    di = wmb.image_desc(din, rows, cols, wmb.ROW_MAJOR, wmb.U8, ld=ls)
    do = wmb.image_desc(dout, rows, cols, wmb.ROW_MAJOR, wmb.U8)
    for mask in (wmb.ME, wmb.NVF):
        a, corr = np.zeros(B, np.float32), np.zeros(B, np.float32)
        wm.embed_batch(0, di, di, do, rows * ls, rows * ls, rows * cols, B, mask, a)
        wm.detect_batch(0, do, rows * cols, B, mask, corr)
        wm.sync(0)
        z = np.zeros((B, rows, cols), np.uint8)
        L.wm_dev_download(wm._h, z.ctypes.data, dout, z.nbytes)
        for b in range(B):
            what = "batch p=%d %dx%d ls=%d mask=%d image %d" % (p, rows, cols, ls, mask, b)
            e, m = _input_planes(wmb, wm, imgs[b], mask)
            check_stats(what, _k({}, ls, cols, rows * ls), sf, W, e, m, float(a[b]))
            check_apply(what, oracle, imgs[b], m, W, float(a[b]), z[b])
            check_detect(what, wmb, wm, oracle, z[b], W, mask, _k({}, cols, cols, rows * cols), float(corr[b]), p=p)
    L.wm_dev_free(wm._h, din)
    L.wm_dev_free(wm._h, dout)
    wm.close()


# ---------------------------------------------------------------------------------------------------
# checks 3-5 on the video driver (wm_process_frames, EMBED_VERIFY, ME): 20 4K frames, the first and the last frame of every run
# ---------------------------------------------------------------------------------------------------
N_VIDEO = 20


def _runs(n, per_run):
    """The video driver's runs of n gated frames (wm_api.cu, wm_process_frames): ceil(n / per_run) runs of even length."""
    nruns = -(-n // per_run)
    base, extra = divmod(n, nruns)
    runs, g = [], 0
    for r in range(nruns):
        nb = base + (1 if r < extra else 0)
        runs.append((g, g + nb - 1))
        g += nb
    return runs


def _video_checks(wmb, oracle, wm, frames, out, sc, runs, tag):
    rows, cols = FULL_4K
    W = _w(rows, cols)
    sf = wm.strength_factor
    k = _k({}, cols, cols)
    checked = sorted({i for r in runs for i in r})
    for i in checked:
        what = "%s frame %d" % (tag, i)
        e, m = _input_planes(wmb, wm, frames[i], wmb.ME)
        check_stats(what, k, sf, W, e, m, float(sc[i]))
        check_apply(what, oracle, frames[i], m, W, float(sc[i]), out[i])
        check_detect(what, wmb, wm, oracle, out[i], W, wmb.ME, k, float(sc[N_VIDEO + i]))
    return checked


@functools.lru_cache(maxsize=None)
def _video_frames():
    rows, cols = FULL_4K
    return np.stack([_frame(rows, cols, 100 + i) for i in range(N_VIDEO)])


def test_video_device_frames_4k(wmb, oracle):
    rows, cols = FULL_4K
    frames = _video_frames()
    wm = _wm(wmb, rows, cols, _w(rows, cols))
    L = wmb.lib()
    dfr = L.wm_dev_alloc(wm._h, frames.nbytes)
    dout = L.wm_dev_alloc(wm._h, frames.nbytes)
    L.wm_dev_upload(wm._h, dfr, frames.ctypes.data, frames.nbytes)
    ctx = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=cols, frames_on_device=True)
    sc = np.zeros(2 * N_VIDEO, np.float32)
    assert wmb.process_frames(ctx, wmb.VIDEO_EMBED_VERIFY, dfr, dout, 0, N_VIDEO, sc) == N_VIDEO
    out = np.zeros_like(frames)
    L.wm_dev_download(wm._h, out.ctypes.data, dout, out.nbytes)
    L.wm_dev_free(wm._h, dfr)
    L.wm_dev_free(wm._h, dout)
    runs = _runs(N_VIDEO, min(32, (136 << 20) // (rows * cols)))  # WM_OPT_RUN_MB = 136: 17 4K frames at most, two runs of 10
    assert len(runs) == 2
    _video_checks(wmb, oracle, wm, frames, out, sc, runs, "video device")
    wm.close()


@pytest.mark.parametrize("padded_upload", [1, 0])
def test_video_host_frames_4k(wmb, oracle, padded_upload):
    rows, cols = FULL_4K
    ls = cols + 64
    frames = _video_frames()
    wm = _wm(wmb, rows, cols, _w(rows, cols), opts={"PADDED_UPLOAD": padded_upload})
    L = wmb.lib()
    nbytes = N_VIDEO * rows * ls
    ptr = L.wm_host_alloc_pinned(nbytes)
    assert ptr
    try:
        host = np.frombuffer((C.c_uint8 * nbytes).from_address(ptr), np.uint8).reshape(N_VIDEO, rows, ls)
        host[:] = 201
        host[:, :, :cols] = frames
        out = np.zeros_like(frames)
        ctx = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=ls, frames_on_device=False)
        sc = np.zeros(2 * N_VIDEO, np.float32)
        assert wmb.process_frames(ctx, wmb.VIDEO_EMBED_VERIFY, ptr, out.ctypes.data, 0, N_VIDEO, sc) == N_VIDEO
        del host
    finally:
        L.wm_host_free_pinned(ptr)
    _video_checks(wmb, oracle, wm, frames, out, sc, _runs(N_VIDEO, 4), "video host padded_upload=%d" % padded_upload)  # 4 frames per run
    wm.close()
