"""ctypes loader for the CPU oracle (oracle/wm_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  The product package
(watermarking-gpu_b200/) never imports this module.

All arrays are row-major (rows, cols) float32, the logical (row, col)
indexing of the reference's af::array (see wm_oracle.c header).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libwm_oracle.so")

ME, NVF = 0, 1


class Opts(C.Structure):
    _fields_ = [("fp16_products", C.c_int), ("sum_f32", C.c_int), ("solve_f32", C.c_int),
                ("contract", C.c_int), ("p", C.c_int), ("rx_f64", C.c_int)]


def opts(fp16_products=1, sum_f32=0, solve_f32=0, contract=1, p=3, rx_f64=0):
    """Canonical (default) = reference-faithful fp16 products, f64 sums/solve, fused mul-add, 3x3 NVF window.
    rx_f64=1: rx() adds every term in f64 (RN16(RN32(x*y)) with fp16_products, the exact x*y without) instead of summing
    64-pixel groups in f32 — a reference without f32 rounding of its own, to bound the GPU's f32 sums by."""
    return Opts(fp16_products, sum_f32, solve_f32, contract, p, rx_f64)


FAITHFUL = opts()
EXACT = opts(fp16_products=0)
STRICT_F32 = opts(sum_f32=1, solve_f32=1)  # every reduction and the LU in f32, like ArrayFire


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE])


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            build()
        L = C.CDLL(_LIB)
        fp = C.POINTER(C.c_float)
        dp = C.POINTER(C.c_double)
        u8p = C.POINTER(C.c_uint8)
        op = C.POINTER(Opts)
        L.wmo_strength.restype = C.c_float
        L.wmo_strength.argtypes = [C.c_float]
        L.wmo_num_threads.restype = C.c_int
        L.wmo_nvf.argtypes = [fp, C.c_int, C.c_int, fp, op]
        L.wmo_rx.argtypes = [fp, C.c_int, C.c_int, op, dp, dp]
        L.wmo_solve8.argtypes = [dp, dp, C.c_int, dp]
        L.wmo_scaled_neighbors.argtypes = [fp, C.c_int, C.c_int, fp, fp, op]
        L.wmo_pred_error_mask.argtypes = [fp, C.c_int, C.c_int, op, fp, fp, fp, dp, dp]
        L.wmo_embed.argtypes = [fp, fp, C.c_int, C.c_int, C.c_int, fp, C.c_float, C.c_int, op, fp, fp,
                                fp, fp, fp]
        L.wmo_apply.argtypes = [fp, fp, C.c_size_t, C.c_float, C.c_int, fp]
        L.wmo_apply.restype = None
        L.wmo_detect.argtypes = [fp, C.c_int, C.c_int, fp, C.c_int, op, fp, fp, fp, fp, fp]
        L.wmo_embed_frame_u8.argtypes = [u8p, C.c_int, C.c_int, C.c_int, fp, C.c_float, C.c_int, op, u8p,
                                         fp]
        L.wmo_detect_frame_u8.argtypes = [u8p, C.c_int, C.c_int, C.c_int, fp, C.c_int, op, fp]
        L.wmo_rgb2gray.argtypes = [fp, C.c_size_t, fp]
        _lib = L
    return _lib


def _f(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(C.POINTER(C.c_float))


def _d(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def num_threads():
    return lib().wmo_num_threads()


def strength(psnr):
    return float(lib().wmo_strength(C.c_float(psnr)))


def nvf(img, o=FAITHFUL):
    img, p = _f(img)
    out = np.empty_like(img)
    lib().wmo_nvf(p, img.shape[0], img.shape[1], out.ctypes.data_as(C.POINTER(C.c_float)), C.byref(o))
    return out


def rx(img, o=FAITHFUL):
    img, p = _f(img)
    Rx = np.zeros(64, np.float64)
    r = np.zeros(8, np.float64)
    lib().wmo_rx(p, img.shape[0], img.shape[1], C.byref(o), _d(Rx), _d(r))
    return Rx.reshape(8, 8), r


def solve8(Rx, r, f32=False):
    Rx = np.ascontiguousarray(Rx, np.float64).reshape(64)
    r = np.ascontiguousarray(r, np.float64)
    c = np.zeros(8, np.float64)
    st = lib().wmo_solve8(_d(Rx), _d(r), int(f32), _d(c))
    return st, c


def scaled_neighbors(img, coef, o=FAITHFUL):
    img, p = _f(img)
    coef, cp = _f(coef)
    out = np.empty_like(img)
    lib().wmo_scaled_neighbors(p, img.shape[0], img.shape[1], cp, out.ctypes.data_as(C.POINTER(C.c_float)),
                               C.byref(o))
    return out


def pred_error_mask(img, o=FAITHFUL, need_mask=True):
    """-> dict(status, e, coef, mask, Rx, rx)"""
    img, p = _f(img)
    fp = C.POINTER(C.c_float)
    e = np.empty_like(img)
    coef = np.zeros(8, np.float32)
    mask = np.empty_like(img) if need_mask else None
    Rx = np.zeros(64, np.float64)
    r = np.zeros(8, np.float64)
    st = lib().wmo_pred_error_mask(p, img.shape[0], img.shape[1], C.byref(o), e.ctypes.data_as(fp),
                                   coef.ctypes.data_as(fp),
                                   mask.ctypes.data_as(fp) if need_mask else None, _d(Rx), _d(r))
    return dict(status=st, e=e, coef=coef, mask=mask, Rx=Rx.reshape(8, 8), rx=r)


def embed(img, W, psnr, mask_type, base=None, o=FAITHFUL):
    """makeWatermark -> dict(status, out, a, mask, u, coef). base: (rows, cols) or (3, rows, cols)."""
    img, p = _f(img)
    W, wp = _f(W)
    if base is None:
        base = img
    base, bp = _f(base)
    ch = 1 if base.ndim == 2 else base.shape[0]
    fp = C.POINTER(C.c_float)
    out = np.empty_like(base)
    mask = np.empty_like(img)
    u = np.empty_like(img)
    coef = np.zeros(8, np.float32)
    a = C.c_float(float("nan"))
    st = lib().wmo_embed(p, bp, ch, img.shape[0], img.shape[1], wp, C.c_float(psnr), mask_type, C.byref(o),
                         out.ctypes.data_as(fp), C.byref(a), mask.ctypes.data_as(fp), u.ctypes.data_as(fp),
                         coef.ctypes.data_as(fp))
    return dict(status=st, out=out, a=a.value, mask=mask, u=u, coef=coef)


def apply(base, u, a, o=FAITHFUL):
    """The apply step of makeWatermark alone (Watermark.cpp:171): clamp(base + u*a, 0, 255) in f32, fused
    like embed() when o.contract.  base and u: arrays of one shape; a: the strength (rounded to f32)."""
    base, bp = _f(base)
    u, up = _f(u)
    if u.shape != base.shape:
        raise ValueError("u has shape %s, base %s" % (u.shape, base.shape))
    out = np.empty_like(base)
    lib().wmo_apply(bp, up, base.size, C.c_float(a), o.contract, out.ctypes.data_as(C.POINTER(C.c_float)))
    return out


def detect(img, W, mask_type, o=FAITHFUL):
    """detectWatermark -> dict(status, corr, ez, u, eu, coef)"""
    img, p = _f(img)
    W, wp = _f(W)
    fp = C.POINTER(C.c_float)
    ez = np.empty_like(img)
    u = np.empty_like(img)
    eu = np.empty_like(img)
    coef = np.zeros(8, np.float32)
    corr = C.c_float(0)
    st = lib().wmo_detect(p, img.shape[0], img.shape[1], wp, mask_type, C.byref(o), C.byref(corr),
                          ez.ctypes.data_as(fp), u.ctypes.data_as(fp), eu.ctypes.data_as(fp),
                          coef.ctypes.data_as(fp))
    return dict(status=st, corr=corr.value, ez=ez, u=u, eu=eu, coef=coef)


def embed_frame_u8(y, W, psnr, mask_type=ME, width=None, o=FAITHFUL):
    """Video path (main.cpp:343-389). y: (height, linesize) uint8, `width` <= linesize the visible
    width (row padding beyond it is skipped); returns (status, out(height, width), a)."""
    y = np.ascontiguousarray(y, np.uint8)
    h = y.shape[0]
    ls = y.shape[1]
    w = ls if width is None else width
    W, wp = _f(W)
    out = np.empty((h, w), np.uint8)
    a = C.c_float(float("nan"))
    u8p = C.POINTER(C.c_uint8)
    st = lib().wmo_embed_frame_u8(y.ctypes.data_as(u8p), ls, h, w, wp, C.c_float(psnr), mask_type,
                                  C.byref(o), out.ctypes.data_as(u8p), C.byref(a))
    return st, out, a.value


def detect_frame_u8(y, W, mask_type=ME, width=None, o=FAITHFUL):
    y = np.ascontiguousarray(y, np.uint8)
    h = y.shape[0]
    ls = y.shape[1]
    w = ls if width is None else width
    W, wp = _f(W)
    corr = C.c_float(0)
    st = lib().wmo_detect_frame_u8(y.ctypes.data_as(C.POINTER(C.c_uint8)), ls, h, w, wp, mask_type,
                                   C.byref(o), C.byref(corr))
    return st, corr.value


def rgb2gray(rgb):
    """rgb: (3, rows, cols) f32 0..255 -> (rows, cols)"""
    rgb, p = _f(rgb)
    n = rgb.shape[1] * rgb.shape[2]
    g = np.empty(rgb.shape[1:], np.float32)
    lib().wmo_rgb2gray(p, n, g.ctypes.data_as(C.POINTER(C.c_float)))
    return g
