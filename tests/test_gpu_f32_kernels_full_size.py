"""The f32 kernels one by one at full frame sizes, in both layouts, each against a reference of its own operation built from the GPU's own
inputs to that kernel (f32_exact.py): the Rx sweep within its derived bound of the f64 sum of the same terms (bit for bit on
integer-valued pixels), the coefficients, the prediction-error and mask planes and the f32 output bit for bit, the stats kernel's sum2
and `a` and the detector's three sums and correlation within their derived bounds.  Every path that runs these kernels on f32 images is
checked on its own: the replayed synchronous calls (gray and RGB base), each option set away from its default, the bench's batch of 148
col-major 1080p images, many small images in one launch, the host-buffer embed-and-verify batch and the video driver on 10-bit frames.

Batched calls sweep an image with fewer CTAs than a single call, and on real-valued pixels the bits of Rx depend on that split.  So the
coefficients a batched image was processed with are taken from a replay: the same image as image 0 of a batch in which image 0 gets as
many sweep CTAs as that image did (f32_exact.sweep_ctas), whose Rx and coefficients the debug interface reports."""
import functools

import numpy as np
import pytest

import f32_exact as X
import util
from test_gpu_parity import report

pytestmark = pytest.mark.gpu

LAYOUTS = [0, 1]  # COL_MAJOR, ROW_MAJOR
SIZE_IDS = ["%dx%d_ld%d" % s for s in X.SIZES]
FULL_4K = (2160, 3840)


def _check(what, observed, bound):
    ratio = observed / bound
    report("f32 full size %s: observed %.3g bound %.3g ratio %.3f" % (what, observed, bound, ratio))
    assert observed <= bound, (what, observed, bound)


def _exact(what, got, want):
    bad = X.unequal(got, want)
    report("f32 full size %s: unequal values %d of %d" % (what, bad, np.asarray(want).size))
    assert bad == 0, (what, np.argwhere(np.asarray(got) != np.asarray(want))[:5].tolist())


def _wm(wmb, rows, cols, W, p=3, opts=None):
    wm = wmb.Watermark(rows, cols, W, p, 40.0)
    for name, v in (opts or {}).items():
        wm.set_option(getattr(wmb, "OPT_" + name), v)
    return wm


@functools.lru_cache(maxsize=None)
def _frame(rows, cols, seed):
    return X.frame(rows, cols, seed)


@functools.lru_cache(maxsize=None)
def _w(rows, cols):
    return util.normal_w(rows, cols)


@functools.lru_cache(maxsize=None)
def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _ld(rows, cols, ld, layout):
    """Row pitch in elements of an image of `layout` carrying the padding of a SIZES entry (0 = dense)."""
    return 0 if not ld else (rows if layout == 0 else cols) + (ld - cols)


def _mem(img, layout):
    """(rows, cols) or (ch, rows, cols) logical image -> its memory order in `layout`."""
    return np.ascontiguousarray(np.swapaxes(img, -1, -2) if layout == 0 else img, np.float32)


def _dev(wmb, wm, img, layout, ld=0):
    """An f32 DeviceArray of `layout` holding img (rows, cols) or (3, rows, cols); its row padding holds 77.0, never to be read."""
    ch = 1 if img.ndim == 2 else img.shape[0]
    rows, cols = img.shape[-2:]
    d = wmb.DeviceArray(wm, rows, cols, layout, wmb.F32, ch, ld)
    buf = np.full((ch, d.L, d.ld), 77.0, np.float32)
    buf[:, :, :d.P] = _mem(img.reshape(ch, rows, cols), layout)
    assert wmb.lib().wm_dev_upload(wm._h, d.ptr, buf.ctypes.data, buf.nbytes) == 0
    return d


def _sums(ez, eu):
    ez, eu = ez.astype(np.float64).ravel(), eu.astype(np.float64).ravel()
    return float(np.dot(eu, ez)), float(np.dot(ez, ez)), float(np.dot(eu, eu))


# ---------------------------------------------------------------------------------------------------
# the checks
# ---------------------------------------------------------------------------------------------------
def check_sweep(what, oracle, f, Rx, rx, coef, mode, f32_solve=False):
    """Check 1: Rx and rx within rx_rel_bound of the f64 sum of the same terms; the coefficients are the LU of the GPU's own system."""
    oRx, orx = oracle.rx(f, oracle.opts(fp16_products=0 if mode == "ffma" else 1, rx_f64=1))
    dev = np.concatenate([(Rx / oRx - 1).ravel(), rx / orx - 1])
    report("f32 full size %s Rx %s: signed relative deviation from %.3g to %.3g" % (what, mode, dev.min(), dev.max()))
    _check("%s Rx %s" % (what, mode), float(np.abs(dev).max()), X.rx_rel_bound(mode, f.size))
    st, oc = oracle.solve8(Rx, rx, f32=f32_solve)
    assert st == 0, what
    _exact("%s coefficients" % what, coef, oc.astype(np.float32))


def check_stats(what, oracle, sf, W, f, c, mask, a, sum2=None, emax=None, p=3):
    """Check 3: `a` (and sum2, max|e| where the call exposes them) against f64 sums over the planes of the GPU's coefficients c."""
    n = W.size
    k = X.chain_len(256)
    x, e = X.stats_input(oracle, f, c, mask, p)
    s_ref = float(np.sum(np.square((x * W).astype(np.float64))))
    nrm = np.sqrt(s_ref)
    if e is not None:
        mx = np.float32(np.abs(e).max())
        if emax is not None:
            assert emax == mx, (what, emax, mx)
        nrm = nrm / float(mx)
    a_ref = sf / (nrm / np.sqrt(float(n)))
    if sum2 is not None:
        _check("%s sum2" % what, abs(sum2 - s_ref), X.sum_rel_bound(k, n) * s_ref)
    _check("%s a" % what, abs(a - a_ref), X.a_rel_bound(k, n) * a_ref)


def check_apply(what, oracle, base, m, W, a, got):
    """Check 4: every plane of the f32 output is the apply step on the GPU's mask plane and `a`, bit for bit; both clamps fire."""
    rows, cols = m.shape
    planes, outs = base.reshape(-1, rows, cols), got.reshape(-1, rows, cols)
    lo = hi = 0
    want = np.empty_like(outs)
    for i in range(planes.shape[0]):
        want[i] = X.apply_ref(oracle, planes[i], m, W, a)[0]
        l, h = X.clamps(planes[i], m, W, a)
        lo, hi = lo + l, hi + h
    report("f32 full size %s apply: clamped at 0: %d, at 255: %d" % (what, lo, hi))
    assert lo > 0 and hi > 0, (what, lo, hi)
    _exact("%s apply output" % what, outs, want)


def check_detect(what, wmb, wm, oracle, z, c, W, mask, corr, sums=None, p=3, layout=1, planes=True):
    """Check 5: the correlation (and the three sums where the call exposes them) against f64 sums of the planes of the watermarked
    image z for the coefficients c of the call.  planes: also run the plane-writing detector on z (3 x 3 masks), whose u and e_u must be
    the planes of its own coefficients bit for bit and whose sums and correlation must meet the same bounds."""
    n = W.size
    k = X.chain_len(256)

    def bounds(tag, c_, corr_, sums_):
        ez, u, eu = X.detect_planes(oracle, z, c_, W, mask, p)
        dot, nz, nu = _sums(ez, eu)
        if sums_ is not None:
            _check("%s dot" % tag, abs(sums_[0] - dot), X.dot_abs_bound(k, n, nz, nu))
            _check("%s nz" % tag, abs(sums_[1] - nz), X.sum_rel_bound(k, n) * nz)
            _check("%s nu" % tag, abs(sums_[2] - nu), X.sum_rel_bound(k, n) * nu)
        _check("%s corr" % tag, abs(corr_ - dot / np.sqrt(nz * nu)), X.corr_abs_bound(k, n, dot, nz, nu))
        return u, eu

    bounds(what, c, corr, sums)
    if planes and (mask == wmb.ME or p == 3):
        dz = _dev(wmb, wm, z, layout)
        ug, eug, corr32 = wm.debug_detect_planes(dz, mask)
        s32, cd = wm.debug(wmb.DBG_SCALARS), wm.debug(wmb.DBG_COEFFS)
        dz.free()
        u, eu = bounds(what + " detector planes", cd, corr32, s32[4:7])
        _exact("%s detector u" % what, ug, u)
        _exact("%s detector e_u" % what, eug, eu)


# ---------------------------------------------------------------------------------------------------
# checks 1 and 2: the Rx sweep, the solve and the planes at full size
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("rows,cols,ld", X.SIZES, ids=SIZE_IDS)
def test_sweep_and_planes(wmb, oracle, rows, cols, ld, layout):
    f = _frame(rows, cols, 31)
    W = _w(rows, cols)
    ldl = _ld(rows, cols, ld, layout)
    tag = "%dx%d ld=%d layout=%d" % (rows, cols, ld, layout)
    wm = _wm(wmb, rows, cols, W)
    d = _dev(wmb, wm, f, layout, ldl)
    wm.detectWatermark(d, wmb.ME)
    check_sweep(tag, oracle, f, wm.debug(wmb.DBG_RX), wm.debug(wmb.DBG_RXVEC), wm.debug(wmb.DBG_COEFFS), "hmma")
    # integer-valued f32 pixels: every partial sum is exact, so Rx is the oracle's bit for bit (a missing tile line shows here at any size)
    fi = np.rint(f)
    di = _dev(wmb, wm, fi, layout, ldl)
    wm.detectWatermark(di, wmb.ME)
    oRx, orx = oracle.rx(fi, oracle.FAITHFUL)
    _exact(tag + " integer-valued Rx", wm.debug(wmb.DBG_RX), oRx)
    _exact(tag + " integer-valued rx", wm.debug(wmb.DBG_RXVEC), orx)
    di.free()
    # the planes, against the oracle's with the coefficients each plane was computed with
    e = wm.debug_plane(d, wmb.DBG_ERRSEQ)
    _exact(tag + " plane errseq", e, X.error_plane(oracle, f, wm.debug(wmb.DBG_COEFFS)))
    m = wm.debug_plane(d, wmb.DBG_MASK_ME)
    _exact(tag + " plane mask_me", m, X.me_mask(X.error_plane(oracle, f, wm.debug(wmb.DBG_COEFFS))))
    _exact(tag + " plane mask_nvf", wm.debug_plane(d, wmb.DBG_MASK_NVF), oracle.nvf(f))
    wm.close()
    wm5 = _wm(wmb, rows, cols, W, p=5)
    d5 = _dev(wmb, wm5, f, layout, ldl)
    _exact(tag + " plane mask_nvf_p5", wm5.debug_plane(d5, wmb.DBG_MASK_NVF), oracle.nvf(f, oracle.opts(p=5)))
    wm5.close()


# ---------------------------------------------------------------------------------------------------
# checks 1 and 3-5 on the synchronous calls (the third call of each is a graph replay), default options and each option set away
# from its default
# ---------------------------------------------------------------------------------------------------
def _sync_checks(wmb, oracle, rows, cols, ld, layout, mask, opts, tag, rgb=True):
    f = _frame(rows, cols, 47)
    W = _w(rows, cols)
    wm = _wm(wmb, rows, cols, W, opts=opts)
    sf = wm.strength_factor
    f32s = bool(opts.get("F32_SOLVE", 0))
    em, dm = X.mode_of(opts)
    what = "%s %dx%d ld=%d layout=%d mask=%d sync" % (tag, rows, cols, ld, layout, mask)
    d = _dev(wmb, wm, f, layout, _ld(rows, cols, ld, layout))
    out = wmb.DeviceArray(wm, rows, cols, layout, wmb.F32)
    for _ in range(3):
        _, a, st = wm.makeWatermark(d, d, mask, out=out)
    assert st == 0
    s = wm.debug(wmb.DBG_SCALARS)
    assert s[1] == np.float32(a)
    c_in = wm.debug(wmb.DBG_COEFFS)
    if mask == wmb.ME:  # the NVF embed runs no sweep
        check_sweep(what + " embed", oracle, f, wm.debug(wmb.DBG_RX), wm.debug(wmb.DBG_RXVEC), c_in, em, f32s)
    z = out.numpy()
    if rgb:
        base = np.stack([_frame(rows, cols, 91 + i) for i in range(3)])
        db = _dev(wmb, wm, base, layout)
        out3 = wmb.DeviceArray(wm, rows, cols, layout, wmb.F32, 3)
        for _ in range(3):
            _, a3, st = wm.makeWatermark(d, db, mask, out=out3)
        assert st == 0 and a3 == a
        z3 = out3.numpy()
    for _ in range(3):
        corr, st = wm.detectWatermark(out, mask)
    assert st == 0
    sd = wm.debug(wmb.DBG_SCALARS)
    c_z = wm.debug(wmb.DBG_COEFFS)
    check_sweep(what + " detect", oracle, z, wm.debug(wmb.DBG_RX), wm.debug(wmb.DBG_RXVEC), c_z, dm, f32s)
    check_stats(what, oracle, sf, W, f, c_in, mask, a, sum2=s[3], emax=s[2] if mask == wmb.ME else None)
    m = X.mask_plane(oracle, f, c_in, mask)
    check_apply(what + " gray", oracle, f, m, W, a, z)
    if rgb:
        check_apply(what + " rgb", oracle, base, m, W, a, z3)
    check_detect(what, wmb, wm, oracle, z, c_z, W, mask, corr, sums=sd[4:7], layout=layout)
    wm.close()


@pytest.mark.parametrize("mask", [0, 1])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("rows,cols,ld", X.SIZES, ids=SIZE_IDS)
def test_sync_calls(wmb, oracle, rows, cols, ld, layout, mask):
    _sync_checks(wmb, oracle, rows, cols, ld, layout, mask, {}, "defaults", rgb=rows * cols <= 1080 * 1920)


OPTIONS = [("USE_TMA", 0), ("TMA_STORE", 0), ("PDL", 0), ("MMA_ACCUM", 0), ("FUSED_SINGLE", 1), ("FP16_PRODUCTS", 0), ("F32_SOLVE", 1)]


@pytest.mark.parametrize("opt,value", OPTIONS, ids=[o for o, _ in OPTIONS])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("rows,cols,ld", [(1080, 1920, 0), (130, 264, 272)], ids=["1080x1920", "130x264_ld272"])
def test_each_option_meets_the_checks(wmb, oracle, rows, cols, ld, layout, opt, value):
    for mask in (wmb.ME, wmb.NVF):
        _sync_checks(wmb, oracle, rows, cols, ld, layout, mask, {opt: value}, "%s=%d" % (opt, value), rgb=False)


# ---------------------------------------------------------------------------------------------------
# batched calls: the coefficients of an image come from a replay with the same sweep split
# ---------------------------------------------------------------------------------------------------
class Replay:
    """Sweeps images as image 0 of a batch (on slot 0) in which image 0 gets a given number of sweep CTAs -> (Rx, rx, coefficients)."""

    def __init__(self, wmb, wm, rows, cols, layout):
        self.wmb, self.wm, self.rows, self.cols, self.layout = wmb, wm, rows, cols, layout
        self.bufs = {}

    def __call__(self, img, nblk):
        wmb, L = self.wmb, self.wmb.lib()
        B = X.replay_batch(nblk, _sms())
        assert B is not None, nblk
        assert X.sweep_ctas(B, X.ntiles(self.rows, self.cols, self.layout == 0), _sms())[0] == nblk
        mem = _mem(img, self.layout)
        if B not in self.bufs:
            self.bufs[B] = L.wm_dev_alloc(self.wm._h, B * mem.nbytes)
            for i in range(1, B):
                L.wm_dev_upload(self.wm._h, self.bufs[B] + i * mem.nbytes, mem.ctypes.data, mem.nbytes)
        ptr = self.bufs[B]
        L.wm_dev_upload(self.wm._h, ptr, mem.ctypes.data, mem.nbytes)
        corr = np.zeros(B, np.float32)
        self.wm.detect_batch(0, wmb.image_desc(ptr, self.rows, self.cols, self.layout, wmb.F32), img.size, B, wmb.ME, corr)
        self.wm.sync(0)
        return self.wm.debug(wmb.DBG_RX), self.wm.debug(wmb.DBG_RXVEC), self.wm.debug(wmb.DBG_COEFFS)

    def free(self):
        for p in self.bufs.values():
            self.wmb.lib().wm_dev_free(self.wm._h, p)


def _batch_image_checks(wmb, oracle, wm, replay, nblk, f, z, W, mask, a, corr, what):
    """Checks 1 and 3-5 of image f of a batch (watermarked z, strength a, correlation of z corr), its sweeps replayed with nblk CTAs."""
    sf = wm.strength_factor
    c_in = None
    if mask == wmb.ME:
        Rx, rx, c_in = replay(f, nblk)
        check_sweep(what + " embed", oracle, f, Rx, rx, c_in, "hmma")
    check_stats(what, oracle, sf, W, f, c_in, mask, a)
    check_apply(what, oracle, f, X.mask_plane(oracle, f, c_in, mask), W, a, z)
    Rz, rz, c_z = replay(z, nblk)
    check_sweep(what + " detect", oracle, z, Rz, rz, c_z, "hmma")
    check_detect(what, wmb, wm, oracle, z, c_z, W, mask, corr, planes=False)


def _stack_frames(rows, cols, B):
    """B real-valued frames: 8 distinct ones, each repeated with a growing non-integer brightness offset."""
    base = [_frame(rows, cols, 700 + k) for k in range(8)]
    return np.stack([np.clip(base[b % 8] + np.float32(0.37 * (b // 8)), 0, 255) for b in range(B)]).astype(np.float32)


def _check_images(nb):
    """Images 0 and B - 1, and the first and last image of each distinct sweep split."""
    picks = {0, len(nb) - 1}
    for v in set(nb):
        idx = [i for i, x in enumerate(nb) if x == v]
        picks |= {idx[0], idx[-1]}
    return sorted(picks)


def test_bench_batch_1080p_col_major(wmb, oracle):
    """bench.py's image1080p call: 148 col-major f32 1080p images per call, NVF then ME embed, NVF and ME detect."""
    rows, cols, B = 1080, 1920, 148
    layout = wmb.COL_MAJOR
    W = _w(rows, cols)
    imgs = _stack_frames(rows, cols, B)
    wm = _wm(wmb, rows, cols, W)
    L = wmb.lib()
    npx = rows * cols
    mem = np.ascontiguousarray(np.swapaxes(imgs, 1, 2))
    din = L.wm_dev_alloc(wm._h, mem.nbytes)
    L.wm_dev_upload(wm._h, din, mem.ctypes.data, mem.nbytes)
    del mem
    douts = {m: L.wm_dev_alloc(wm._h, imgs.nbytes) for m in (wmb.NVF, wmb.ME)}
    di = wmb.image_desc(din, rows, cols, layout, wmb.F32)
    res = {}
    for mask in (wmb.NVF, wmb.ME):
        a = np.zeros(B, np.float32)
        wm.embed_batch(0, di, di, wmb.image_desc(douts[mask], rows, cols, layout, wmb.F32), npx, npx, npx, B, mask, a)
        res[mask] = [a]
    for mask in (wmb.NVF, wmb.ME):
        corr = np.zeros(B, np.float32)
        wm.detect_batch(0, wmb.image_desc(douts[mask], rows, cols, layout, wmb.F32), npx, B, mask, corr)
        res[mask].append(corr)
    wm.sync(0)
    nb = X.sweep_ctas(B, X.ntiles(rows, cols, True), _sms())
    picks = _check_images(nb)
    report("f32 full size bench batch: sweep CTAs per image %s, checked images %s" % (sorted(set(nb)), picks))
    replay = Replay(wmb, wm, rows, cols, layout)
    for mask in (wmb.NVF, wmb.ME):
        a, corr = res[mask]
        for b in picks:
            zm = np.empty((cols, rows), np.float32)
            L.wm_dev_download(wm._h, zm.ctypes.data, douts[mask] + b * 4 * npx, zm.nbytes)
            _batch_image_checks(wmb, oracle, wm, replay, nb[b], imgs[b], np.ascontiguousarray(zm.T), W, mask, float(a[b]), float(corr[b]),
                                "bench batch mask=%d image %d" % (mask, b))
    replay.free()
    for p in [din] + list(douts.values()):
        L.wm_dev_free(wm._h, p)
    wm.close()


def test_many_small_images_one_launch(wmb, oracle):
    """320 small row-major images in one launch sequence: one or two sweep CTAs per image (the frame ring's thread-per-pixel mode)."""
    rows, cols, B = 96, 160, 320
    W = _w(rows, cols)
    imgs = _stack_frames(rows, cols, B)
    wm = _wm(wmb, rows, cols, W)
    L = wmb.lib()
    n = rows * cols
    din, dout = L.wm_dev_alloc(wm._h, imgs.nbytes), L.wm_dev_alloc(wm._h, imgs.nbytes)
    L.wm_dev_upload(wm._h, din, imgs.ctypes.data, imgs.nbytes)
    di = wmb.image_desc(din, rows, cols, wmb.ROW_MAJOR, wmb.F32)
    do = wmb.image_desc(dout, rows, cols, wmb.ROW_MAJOR, wmb.F32)
    a, c, st = np.zeros(B, np.float32), np.zeros(B, np.float32), np.zeros(B, np.int32)
    wm.embed_batch(0, di, di, do, n, n, n, B, wmb.ME, a, st)
    wm.detect_batch(0, do, n, B, wmb.ME, c, st)
    wm.sync(0)
    outs = np.zeros_like(imgs)
    L.wm_dev_download(wm._h, outs.ctypes.data, dout, outs.nbytes)
    nb = X.sweep_ctas(B, X.ntiles(rows, cols, False), _sms())
    picks = _check_images(nb)
    report("f32 full size many small: sweep CTAs per image %s, checked images %s" % (sorted(set(nb)), picks))
    replay = Replay(wmb, wm, rows, cols, wmb.ROW_MAJOR)
    for b in picks:
        _batch_image_checks(wmb, oracle, wm, replay, nb[b], imgs[b], outs[b], W, wmb.ME, float(a[b]), float(c[b]), "many small image %d" % b)
    replay.free()
    L.wm_dev_free(wm._h, din)
    L.wm_dev_free(wm._h, dout)
    wm.close()


@pytest.mark.parametrize("layout", LAYOUTS)
def test_embed_verify_host_batch_1080p(wmb, oracle, layout):
    rows, cols, B = 1080, 1920, 2
    W = _w(rows, cols)
    imgs = _stack_frames(rows, cols, B)
    wm = _wm(wmb, rows, cols, W)
    hin = _mem(imgs, layout)
    hout = np.zeros_like(hin)
    n = rows * cols
    di = wmb.image_desc(hin.ctypes.data, rows, cols, layout, wmb.F32)
    do = wmb.image_desc(hout.ctypes.data, rows, cols, layout, wmb.F32)
    nb = X.sweep_ctas(B, X.ntiles(rows, cols, layout == 0), _sms())
    replay = Replay(wmb, wm, rows, cols, layout)
    for mask in (wmb.ME, wmb.NVF):
        a, corr, st = np.zeros(B, np.float32), np.zeros(B, np.float32), np.zeros(B, np.int32)
        wm.embed_verify_host_batch(1, di, di, do, n, n, n, B, mask, a, corr, st)
        wm.sync(1)
        assert np.all(st == 0)
        for b in range(B):
            z = np.ascontiguousarray(hout[b].T) if layout == 0 else hout[b]
            _batch_image_checks(wmb, oracle, wm, replay, nb[b], imgs[b], z, W, mask, float(a[b]), float(corr[b]),
                                "host verify layout=%d mask=%d image %d" % (layout, mask, b))
    replay.free()
    wm.close()


# ---------------------------------------------------------------------------------------------------
# the video driver on 10-bit 4K frames (WM_Y10, EMBED_VERIFY): the f32 kernels on x = v / 4
# ---------------------------------------------------------------------------------------------------
def test_video_y10_4k_embed_verify(wmb, oracle):
    """8 device frames in runs of 4 (WM_OPT_RUN_MB = 64: every frame of a run gets the same number of sweep CTAs); the first and the
    last frame of each run.  Output words: (uint16) clamp(4 y, 0, 1023) of the apply step on x with the mask plane of the run's
    coefficients and the driver's own `a`, no difference allowed; `a` and the correlation of x' = v' / 4 within their bounds."""
    from test_gpu_y10 import samples
    rows, cols = FULL_4K
    n = 8
    W = _w(rows, cols)
    v = np.stack([samples(rows, cols, seed=120 + i) for i in range(n)])
    wm = _wm(wmb, rows, cols, W, opts={"RUN_MB": 64})
    L = wmb.lib()
    words = np.ascontiguousarray(v.astype("<u2"))
    dfr, dout = L.wm_dev_alloc(wm._h, words.nbytes), L.wm_dev_alloc(wm._h, words.nbytes)
    L.wm_dev_upload(wm._h, dfr, words.ctypes.data, words.nbytes)
    ctx = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=2 * cols, frames_on_device=True, layout=wmb.Y10)
    sc = np.zeros(2 * n, np.float32)
    assert wmb.process_frames(ctx, wmb.VIDEO_EMBED_VERIFY, dfr, dout, 0, n, sc) == n
    out = np.zeros_like(words)
    L.wm_dev_download(wm._h, out.ctypes.data, dout, out.nbytes)
    L.wm_dev_free(wm._h, dfr)
    L.wm_dev_free(wm._h, dout)
    per_run = (64 << 20) // (rows * 2 * cols)
    assert per_run == 4
    nb = X.sweep_ctas(per_run, X.ntiles(rows, cols, False), _sms())
    assert len(set(nb)) == 1
    replay = Replay(wmb, wm, rows, cols, wmb.ROW_MAJOR)
    sf = wm.strength_factor
    for i in (0, 3, 4, 7):
        what = "video y10 frame %d" % i
        x = v[i].astype(np.float32) * np.float32(0.25)
        a = float(sc[i])
        Rx, rx, c = replay(x, nb[0])
        check_sweep(what + " embed", oracle, x, Rx, rx, c, "hmma")
        check_stats(what, oracle, sf, W, x, c, wmb.ME, a)
        m = X.mask_plane(oracle, x, c, wmb.ME)
        y, _ = X.apply_ref(oracle, x, m, W, a)
        lo, hi = X.clamps(x, m, W, a)
        report("f32 full size %s apply: clamped at 0: %d, at 255: %d" % (what, lo, hi))
        _exact(what + " output words", out[i].astype(np.uint16), X.y10_words(y))
        xz = (out[i] & 0x3FF).astype(np.float32) * np.float32(0.25)
        Rz, rz, cz = replay(xz, nb[0])
        check_sweep(what + " detect", oracle, xz, Rz, rz, cz, "hmma")
        check_detect(what, wmb, wm, oracle, xz, cz, W, wmb.ME, float(sc[n + i]), planes=False)
    replay.free()
    wm.close()
