"""watermarking-gpu_b200 — Python host mirror of the reference's `Watermark` class over the C ABI.

The product is libwm_b200.so (hand-written sm_100a CUDA behind include/wm_b200.h) and the C++ façade
csrc/Watermark.hpp.  This module is plumbing for tests and bench.py: a ctypes binding whose `Watermark`
class keeps the reference's surface (Watermark_GPU/Watermark.hpp:62-71: makeWatermark / detectWatermark with
ME and NVF mask types, same image / W / p / psnr inputs, `a` and correlation outputs).

There is NO CPU fallback here: if the CUDA library is missing or no GPU is present, calls raise.
Nothing in this package imports oracle/.
"""
import ctypes as C
import importlib.util
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libwm_b200.so")

ME, NVF = 0, 1                      # Watermark.hpp:10-14
COL_MAJOR, ROW_MAJOR = 0, 1
PACKED_RGB, PACKED_BGR = 2, 3       # interleaved 8-bit colour (rows, cols, 3), row pitch in bytes
PACKED_RGBA, PACKED_BGRA = 4, 5     # the same with a fourth byte per pixel (rows, cols, 4), copied through by the embed
PACKED_YUYV, PACKED_UYVY = 6, 7     # packed 4:2:2 (rows, cols, 2): luma at [..., 0] / [..., 1], chroma copied through by the embed
Y10, Y10_MSB = 10, 11               # 10-bit luma (rows, cols) uint16: the sample in bits 0-9 (yuv420p10le Y) / 6-15 (P010 Y)
WORD_LAYOUTS = (Y10, Y10_MSB)       # one little-endian 16-bit word per pixel
PACKED_V210 = 12                    # 10-bit 4:2:2 v210 (rows, >= v210_pitch(cols)) uint8: the bytes of its rows, chroma copied through by the embed
PACKED_BYTES = {PACKED_RGB: 3, PACKED_BGR: 3, PACKED_RGBA: 4, PACKED_BGRA: 4, PACKED_YUYV: 2, PACKED_UYVY: 2, Y10: 2, Y10_MSB: 2}  # bytes per pixel of each packed layout
F32, U8 = 0, 1


def v210_pitch(cols):
    """Bytes of a v210 row of `cols` pixels (WM_V210_PITCH): whole 128-byte blocks of 48 pixels."""
    return (cols + 47) // 48 * 128


def row_bytes(layout, cols):
    """Bytes of a row of `cols` pixels of a packed layout (v210: its pitch)."""
    return v210_pitch(cols) if layout == PACKED_V210 else PACKED_BYTES[layout] * cols


OK, SINGULAR, ZERO_MASK = 0, 1, 2
OPT_FP16_PRODUCTS, OPT_KERNEL_TIMING, OPT_USE_TMA, OPT_SERIAL_SLOTS, OPT_CUDA_GRAPHS, OPT_MMA_ACCUM, OPT_SPLIT_COST = 1, 2, 3, 4, 5, 6, 7
OPT_F32_SOLVE, OPT_HOST_RUN_FRAMES, OPT_TMA_STORE, OPT_PDL, OPT_FUSED_SINGLE, OPT_PADDED_UPLOAD, OPT_NARROW_U8, OPT_RUN_MB = 8, 9, 10, 11, 12, 13, 14, 15
DBG_RX, DBG_RXVEC, DBG_COEFFS, DBG_SCALARS, DBG_ERRSEQ, DBG_MASK_NVF, DBG_PHASES, DBG_MASK_ME = range(8)
KERNEL_NAMES = ["rx_sweep", "me_stats", "nvf_stats", "me_apply", "me_detect", "nvf_apply", "nvf_detect"]
VIDEO_EMBED, VIDEO_DETECT, VIDEO_EMBED_VERIFY = 0, 1, 2

# every symbol include/wm_b200.h declares (tests check the .so exports all of them)
EXPORTS = [
    "wm_create", "wm_create_from_file", "wm_clone", "wm_reinitialize", "wm_reinitialize_from_file", "wm_destroy",
    "wm_set_option", "wm_last_error", "wm_strength_factor", "wm_embed", "wm_detect", "wm_num_slots", "wm_get_stream",
    "wm_embed_batch", "wm_detect_batch", "wm_sync", "wm_embed_host", "wm_detect_host", "wm_embed_host_batch",
    "wm_detect_host_batch", "wm_embed_verify_host_batch", "wm_shard_frames", "wm_process_frames_multi", "wm_rgb2gray", "wm_debug_get",
    "wm_debug_set_coeffs", "wm_debug_plane", "wm_debug_detect_planes", "wm_get_kernel_times", "wm_launch_count", "wm_process_frames",
    "wm_dev_alloc", "wm_dev_free", "wm_dev_upload", "wm_dev_download", "wm_host_alloc_pinned",
    "wm_host_free_pinned", "wm_device_count", "wm_version",
]


class wm_image(C.Structure):
    _fields_ = [("data", C.c_void_p), ("rows", C.c_int64), ("cols", C.c_int64), ("ld", C.c_int64),
                ("channels", C.c_int32), ("layout", C.c_int32), ("dtype", C.c_int32), ("reserved", C.c_int32),
                ("plane_stride", C.c_int64)]


class wm_video_ctx(C.Structure):
    _fields_ = [("watermark", C.c_void_p), ("height", C.c_int32), ("width", C.c_int32),
                ("watermark_interval", C.c_int32), ("linesize", C.c_int32), ("frame_stride", C.c_int64),
                ("frames_on_device", C.c_int32), ("layout", C.c_int32)]


class WatermarkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("wm_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def build(force=False):
    spec = importlib.util.spec_from_file_location("_wm_build", os.path.join(_HERE, "build.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    m.build(force=force)
    return m


def lib():
    """Load libwm_b200.so (building it in-tree if absent).  Raises if it cannot be had: no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        build()
    L = C.CDLL(LIB_PATH)
    vp, i64, i32, fp, ip = C.c_void_p, C.c_int64, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int)
    imp = C.POINTER(wm_image)
    L.wm_create.argtypes = [C.POINTER(vp), i64, i64, fp, i32, C.c_float, i32, vp]
    L.wm_create_from_file.argtypes = [C.POINTER(vp), i64, i64, C.c_char_p, i32, C.c_float, i32, vp]
    L.wm_clone.argtypes = [vp, C.POINTER(vp)]
    L.wm_reinitialize.argtypes = [vp, i64, i64, fp]
    L.wm_reinitialize_from_file.argtypes = [vp, i64, i64, C.c_char_p]
    L.wm_destroy.argtypes = [vp]
    L.wm_destroy.restype = None
    L.wm_set_option.argtypes = [vp, i32, i32]
    L.wm_last_error.argtypes = [vp]
    L.wm_last_error.restype = C.c_char_p
    L.wm_strength_factor.argtypes = [vp]
    L.wm_strength_factor.restype = C.c_float
    L.wm_embed.argtypes = [vp, imp, imp, imp, i32, fp]
    L.wm_detect.argtypes = [vp, imp, i32, fp]
    L.wm_num_slots.argtypes = [vp]
    L.wm_get_stream.argtypes = [vp, i32]
    L.wm_get_stream.restype = vp
    L.wm_embed_batch.argtypes = [vp, i32, imp, imp, imp, i64, i64, i64, i32, i32, fp, ip]
    L.wm_detect_batch.argtypes = [vp, i32, imp, i64, i32, i32, fp, ip]
    L.wm_sync.argtypes = [vp, i32]
    L.wm_embed_host.argtypes = [vp, imp, imp, imp, i32, fp]
    L.wm_detect_host.argtypes = [vp, imp, i32, fp]
    L.wm_embed_host_batch.argtypes = [vp, i32, imp, imp, imp, i64, i64, i64, i32, i32, fp, ip]
    L.wm_detect_host_batch.argtypes = [vp, i32, imp, i64, i32, i32, fp, ip]
    L.wm_embed_verify_host_batch.argtypes = [vp, i32, imp, imp, imp, i64, i64, i64, i32, i32, fp, fp, ip]
    L.wm_shard_frames.argtypes = [i64, i32, i32, C.POINTER(i64), C.POINTER(i64)]
    L.wm_shard_frames.restype = None
    L.wm_process_frames_multi.argtypes = [C.POINTER(C.POINTER(wm_video_ctx)), i32, i32, C.POINTER(vp), C.POINTER(vp), i64, i64, fp]
    L.wm_process_frames_multi.restype = i64
    L.wm_rgb2gray.argtypes = [vp, imp, imp, C.c_float, C.c_float, C.c_float]
    L.wm_debug_get.argtypes = [vp, i32, vp]
    L.wm_debug_set_coeffs.argtypes = [vp, fp]
    L.wm_debug_plane.argtypes = [vp, imp, i32, vp]
    L.wm_debug_detect_planes.argtypes = [vp, imp, i32, vp, vp, fp]
    L.wm_get_kernel_times.argtypes = [vp, i32, C.POINTER(C.c_double), i32]
    L.wm_get_kernel_times.restype = i64
    L.wm_launch_count.argtypes = [vp]
    L.wm_launch_count.restype = i64
    L.wm_process_frames.argtypes = [C.POINTER(wm_video_ctx), i32, vp, vp, i64, i64, fp]
    L.wm_process_frames.restype = i64
    L.wm_dev_alloc.argtypes = [vp, i64]
    L.wm_dev_alloc.restype = vp
    L.wm_dev_free.argtypes = [vp, vp]
    L.wm_dev_free.restype = None
    L.wm_dev_upload.argtypes = [vp, vp, vp, i64]
    L.wm_dev_download.argtypes = [vp, vp, vp, i64]
    L.wm_host_alloc_pinned.argtypes = [i64]
    L.wm_host_alloc_pinned.restype = vp
    L.wm_host_free_pinned.argtypes = [vp]
    L.wm_host_free_pinned.restype = None
    L.wm_device_count.restype = i32
    L.wm_version.restype = C.c_char_p
    _lib = L
    return L


def device_count():
    return lib().wm_device_count()


def image_desc(ptr, rows, cols, layout=COL_MAJOR, dtype=F32, ld=0, channels=1, plane_stride=0):
    """wm_image over a raw pointer (device pointer for the device API, host pointer for *_host)."""
    return wm_image(C.c_void_p(ptr), rows, cols, ld, channels, layout, dtype, 0, plane_stride)


_NP_DT = {F32: np.float32, U8: np.uint8}


def _dtype_code(a):
    if a.dtype == np.float32:
        return F32
    if a.dtype == np.uint8:
        return U8
    raise TypeError("images must be float32 or uint8, got %s" % a.dtype)


class DeviceArray:
    """A device buffer holding an image (rows, cols[, 3]) in a given layout; owned via the C ABI.

    Planar layouts hold (rows, cols) or (3, rows, cols) images, `ld` in elements.  The packed layouts hold a (rows, cols, n) uint8
    image, n = PACKED_BYTES[layout], as interleaved rows of n * cols bytes with a row pitch of `ld` bytes (0 = dense); the 10-bit layouts
    (WORD_LAYOUTS) a (rows, cols) uint16 image, as rows of little-endian words; PACKED_V210 a (rows, >= v210_pitch(cols)) uint8 array of
    the bytes of its rows, of which the first v210_pitch(cols) are the row (`ld` bytes apart on the device, 0 = the pitch)."""

    def __init__(self, wm, rows, cols, layout=COL_MAJOR, dtype=F32, channels=1, ld=0):
        packed = layout in PACKED_BYTES or layout == PACKED_V210
        if packed:
            dtype, channels = U8, PACKED_BYTES.get(layout, 0)
        self.wm, self.rows, self.cols, self.layout, self.dtype, self.channels = wm, rows, cols, layout, dtype, channels
        P = rows if layout == COL_MAJOR else cols
        Ln = cols if layout == COL_MAJOR else rows
        if packed:
            P = row_bytes(layout, cols)  # bytes of a row
        self.ld = ld if ld else P
        self.P, self.L = P, Ln
        self.itemsize = 4 if dtype == F32 else 1
        planes = 1 if packed else self.channels
        self.nbytes = planes * Ln * self.ld * self.itemsize
        self.ptr = lib().wm_dev_alloc(wm._h, self.nbytes)
        if not self.ptr:
            raise WatermarkError(-6, "cudaMalloc of %d bytes failed" % self.nbytes)

    @classmethod
    def from_numpy(cls, wm, img, layout=COL_MAJOR, ld=0):
        """img: (rows, cols) or (3, rows, cols) numpy array in logical (row, col) indexing; (rows, cols, PACKED_BYTES[layout]) uint8
        for a packed layout; (rows, >= v210_pitch(wm.cols)) uint8 for PACKED_V210, an image of the watermark's width."""
        img = np.asarray(img)
        if layout == PACKED_V210:
            d = cls(wm, img.shape[0], wm.cols, layout, ld=ld)
            d.upload(img)
            return d
        if layout in PACKED_BYTES:
            d = cls(wm, img.shape[0], img.shape[1], layout, ld=ld)
            d.upload(img)
            return d
        ch = 1 if img.ndim == 2 else img.shape[0]
        rows, cols = img.shape[-2:]
        d = cls(wm, rows, cols, layout, _dtype_code(img), ch, ld)
        d.upload(img)
        return d

    def _to_mem(self, img):
        if self.layout == PACKED_V210:
            buf = np.zeros((self.L, self.ld), np.uint8)
            buf[:, :self.P] = np.asarray(img, np.uint8).reshape(self.rows, -1)[:, :self.P]
            return buf
        if self.layout in WORD_LAYOUTS:
            img = np.ascontiguousarray(np.asarray(img).astype("<u2", casting="same_kind")).view(np.uint8)
        if self.layout in PACKED_BYTES:
            buf = np.zeros((self.L, self.ld), np.uint8)
            buf[:, :self.P] = img.reshape(self.rows, self.P)
            return buf
        planes = img.reshape(self.channels, self.rows, self.cols)
        buf = np.zeros((self.channels, self.L, self.ld), _NP_DT[self.dtype])
        for c in range(self.channels):
            buf[c, :, :self.P] = planes[c].T if self.layout == COL_MAJOR else planes[c]
        return buf

    def upload(self, img):
        img = np.asarray(img) if self.layout in WORD_LAYOUTS else np.asarray(img, _NP_DT[self.dtype])
        buf = np.ascontiguousarray(self._to_mem(img))
        rc = lib().wm_dev_upload(self.wm._h, self.ptr, buf.ctypes.data, buf.nbytes)
        if rc:
            raise WatermarkError(rc, "upload failed")

    def numpy(self):
        if self.layout in PACKED_BYTES or self.layout == PACKED_V210:
            buf = np.empty((self.L, self.ld), np.uint8)
            rc = lib().wm_dev_download(self.wm._h, buf.ctypes.data, self.ptr, buf.nbytes)
            if rc:
                raise WatermarkError(rc, "download failed")
            px = np.ascontiguousarray(buf[:, :self.P])
            if self.layout in WORD_LAYOUTS:
                return px.view("<u2").astype(np.uint16).reshape(self.rows, self.cols)
            if self.layout == PACKED_V210:
                return px
            return px.reshape(self.rows, self.cols, self.channels)
        buf = np.empty((self.channels, self.L, self.ld), _NP_DT[self.dtype])
        rc = lib().wm_dev_download(self.wm._h, buf.ctypes.data, self.ptr, buf.nbytes)
        if rc:
            raise WatermarkError(rc, "download failed")
        v = buf[:, :, :self.P]
        out = np.stack([p.T if self.layout == COL_MAJOR else p for p in v])
        return np.ascontiguousarray(out[0] if self.channels == 1 else out)

    def desc(self):
        return image_desc(self.ptr, self.rows, self.cols, self.layout, self.dtype, self.ld, self.channels, 0)

    def free(self):
        if self.ptr:
            lib().wm_dev_free(self.wm._h, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Watermark:
    """Mirror of the reference's Watermark class (Watermark.hpp:26-71) on the B200 path.

    Watermark(rows, cols, randomMatrixPath_or_array, p, psnr): `randomMatrix` is a path to the raw float32
    row-major W file (Watermark.cpp:62-75) or a (rows, cols) float32 array.
    """

    def __init__(self, rows, cols, random_matrix, p, psnr, device=0, stream=None):
        self._h = None
        h = C.c_void_p()
        L = lib()
        if isinstance(random_matrix, (str, bytes, os.PathLike)):
            rc = L.wm_create_from_file(C.byref(h), rows, cols, os.fsencode(random_matrix), p, psnr, device, stream)
        else:
            w = np.ascontiguousarray(random_matrix, np.float32)
            if w.size != rows * cols:
                raise WatermarkError(-3, "W has %d elements, image is %dx%d" % (w.size, rows, cols))
            rc = L.wm_create(C.byref(h), rows, cols, w.ctypes.data_as(C.POINTER(C.c_float)), p, psnr, device, stream)
        if rc:
            raise WatermarkError(rc, L.wm_last_error(None).decode())
        self._h = h
        self.rows, self.cols, self.p, self.psnr, self.device = rows, cols, p, psnr, device

    # -- lifetime ------------------------------------------------------------------------------
    def clone(self):
        """Copy constructor (Watermark.cpp:30-34): shares W, owns its workspace."""
        h = C.c_void_p()
        self._check(lib().wm_clone(self._h, C.byref(h)))
        o = object.__new__(Watermark)
        o._h, o.rows, o.cols, o.p, o.psnr, o.device = h, self.rows, self.cols, self.p, self.psnr, self.device
        return o

    def reinitialize(self, random_matrix, rows, cols):
        """Watermark.cpp:78-85 (argument order as the reference)."""
        if isinstance(random_matrix, (str, bytes, os.PathLike)):
            rc = lib().wm_reinitialize_from_file(self._h, rows, cols, os.fsencode(random_matrix))
        else:
            w = np.ascontiguousarray(random_matrix, np.float32)
            if w.size != rows * cols:
                raise WatermarkError(-3, "W has %d elements, image is %dx%d" % (w.size, rows, cols))
            rc = lib().wm_reinitialize(self._h, rows, cols, w.ctypes.data_as(C.POINTER(C.c_float)))
        self._check(rc)
        self.rows, self.cols = rows, cols

    def close(self):
        if self._h:
            lib().wm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise WatermarkError(rc, lib().wm_last_error(self._h).decode())
        return rc

    def set_option(self, opt, value):
        self._check(lib().wm_set_option(self._h, opt, int(value)))

    @property
    def strength_factor(self):
        return lib().wm_strength_factor(self._h)

    # -- hot path, device arrays -------------------------------------------------------------------
    def makeWatermark(self, input_image, output_image, mask_type, out=None, out_dtype=None):
        """Watermark.cpp:156-172.  input_image: gray DeviceArray; output_image: gray or RGB DeviceArray (base).
        Returns (watermarked DeviceArray, a, status)."""
        base = output_image if output_image is not None else input_image
        if out is None:
            out = DeviceArray(self, base.rows, base.cols, base.layout, base.dtype if out_dtype is None else out_dtype,
                              base.channels)
        a = C.c_float(float("nan"))
        di, db, do = input_image.desc(), base.desc(), out.desc()
        rc = self._check(lib().wm_embed(self._h, C.byref(di), C.byref(db), C.byref(do), mask_type, C.byref(a)))
        return out, a.value, rc

    def detectWatermark(self, watermarked_image, mask_type):
        """Watermark.cpp:234-250 -> (correlation, status)"""
        corr = C.c_float(0.0)
        d = watermarked_image.desc()
        rc = self._check(lib().wm_detect(self._h, C.byref(d), mask_type, C.byref(corr)))
        return corr.value, rc

    def rgb2gray(self, rgb, weights=(0.299, 0.587, 0.114)):
        """af::rgb2gray with the reference's weights (main.cpp:142-154): RGB DeviceArray -> gray DeviceArray."""
        gray = DeviceArray(self, rgb.rows, rgb.cols, rgb.layout, F32, 1)
        di, do = rgb.desc(), gray.desc()
        self._check(lib().wm_rgb2gray(self._h, C.byref(di), C.byref(do), *[C.c_float(w) for w in weights]))
        return gray

    # -- hot path, host (numpy) arrays: H2D + compute + D2H inside the call -------------------------
    def _host_desc(self, arr, layout):
        if layout == PACKED_V210:  # (rows, >= pitch) uint8, the bytes of each row contiguous; rows may be pitched
            if arr.dtype != np.uint8 or arr.ndim != 2 or arr.strides[1] != 1 or arr.shape[1] < v210_pitch(self.cols):
                raise TypeError("a v210 host image is a (rows, >= v210_pitch(cols)) uint8 array with contiguous rows")
            return image_desc(arr.ctypes.data, self.rows, self.cols, layout, U8, arr.strides[0], 0, 0)
        if layout in WORD_LAYOUTS:  # (rows, cols) uint16, pixels contiguous; rows may be pitched
            if arr.dtype != np.uint16 or arr.ndim != 2 or arr.strides[1] != 2:
                raise TypeError("an image of a 10-bit layout is a (rows, cols) uint16 array with contiguous pixels")
            return image_desc(arr.ctypes.data, self.rows, self.cols, layout, U8, arr.strides[0], 2, 0)
        if layout in PACKED_BYTES:  # (rows, cols, n) uint8, pixels and channels contiguous; rows may be pitched (a view of a wider buffer)
            n = PACKED_BYTES[layout]
            if arr.dtype != np.uint8 or arr.ndim != 3 or arr.shape[2] != n or arr.strides[1:] != (n, 1):
                raise TypeError("a packed host image of this layout is a (rows, cols, %d) uint8 array with contiguous pixels" % n)
            return image_desc(arr.ctypes.data, self.rows, self.cols, layout, U8, arr.strides[0], n, 0)
        ch = 1 if arr.ndim == 2 else arr.shape[0]
        return image_desc(arr.ctypes.data, self.rows, self.cols, layout, _dtype_code(arr), 0, ch, 0)

    def make_watermark_host(self, image_mem, base_mem, out_mem, mask_type, layout=ROW_MAJOR):
        """image_mem/base_mem/out_mem: C-contiguous numpy buffers ALREADY in `layout` memory order
        ((rows, cols) for ROW_MAJOR, (cols, rows) for COL_MAJOR; leading 3 for RGB).  Returns (a, status)."""
        a = C.c_float(float("nan"))
        di = self._host_desc(image_mem, layout)
        db = self._host_desc(base_mem if base_mem is not None else image_mem, layout)
        do = self._host_desc(out_mem, layout)
        rc = self._check(lib().wm_embed_host(self._h, C.byref(di), C.byref(db), C.byref(do), mask_type, C.byref(a)))
        return a.value, rc

    def detect_watermark_host(self, image_mem, mask_type, layout=ROW_MAJOR):
        corr = C.c_float(0.0)
        d = self._host_desc(image_mem, layout)
        rc = self._check(lib().wm_detect_host(self._h, C.byref(d), mask_type, C.byref(corr)))
        return corr.value, rc

    def embed_host_batch(self, slot, in_desc, base_desc, out_desc, in_stride, base_stride, out_stride, batch, mask_type,
                         a_out, status_out=None):
        """Pipelined host-buffer form (descs over HOST pointers); results and output images are valid after sync(slot)."""
        self._check(lib().wm_embed_host_batch(
            self._h, slot, C.byref(in_desc), C.byref(base_desc), C.byref(out_desc), in_stride, base_stride, out_stride,
            batch, mask_type, a_out.ctypes.data_as(C.POINTER(C.c_float)),
            status_out.ctypes.data_as(C.POINTER(C.c_int)) if status_out is not None else None))

    def embed_verify_host_batch(self, slot, in_desc, base_desc, out_desc, in_stride, base_stride, out_stride, batch, mask_type,
                                a_out, corr_out, status_out=None):
        """embed_host_batch + detection of the watermarked images where they lie on the device (one upload, one download per image)."""
        self._check(lib().wm_embed_verify_host_batch(
            self._h, slot, C.byref(in_desc), C.byref(base_desc), C.byref(out_desc), in_stride, base_stride, out_stride,
            batch, mask_type, a_out.ctypes.data_as(C.POINTER(C.c_float)), corr_out.ctypes.data_as(C.POINTER(C.c_float)),
            status_out.ctypes.data_as(C.POINTER(C.c_int)) if status_out is not None else None))

    def detect_host_batch(self, slot, img_desc, img_stride, batch, mask_type, corr_out, status_out=None):
        self._check(lib().wm_detect_host_batch(
            self._h, slot, C.byref(img_desc), img_stride, batch, mask_type,
            corr_out.ctypes.data_as(C.POINTER(C.c_float)),
            status_out.ctypes.data_as(C.POINTER(C.c_int)) if status_out is not None else None))

    # -- batched / pipelined ----------------------------------------------------------------------
    def embed_batch(self, slot, in_desc, base_desc, out_desc, in_stride, base_stride, out_stride, batch, mask_type,
                    a_out, status_out=None):
        """Asynchronous on `slot`; a_out / status_out are numpy arrays that must stay alive until sync()."""
        self._check(lib().wm_embed_batch(
            self._h, slot, C.byref(in_desc), C.byref(base_desc), C.byref(out_desc), in_stride, base_stride, out_stride,
            batch, mask_type, a_out.ctypes.data_as(C.POINTER(C.c_float)),
            status_out.ctypes.data_as(C.POINTER(C.c_int)) if status_out is not None else None))

    def detect_batch(self, slot, img_desc, img_stride, batch, mask_type, corr_out, status_out=None):
        self._check(lib().wm_detect_batch(
            self._h, slot, C.byref(img_desc), img_stride, batch, mask_type,
            corr_out.ctypes.data_as(C.POINTER(C.c_float)),
            status_out.ctypes.data_as(C.POINTER(C.c_int)) if status_out is not None else None))

    def sync(self, slot=-1):
        return self._check(lib().wm_sync(self._h, slot))

    @property
    def num_slots(self):
        return lib().wm_num_slots(self._h)

    def stream(self, slot):
        """cudaStream_t (as int) of a slot, e.g. for torch.cuda.ExternalStream: order your own copies on it."""
        return lib().wm_get_stream(self._h, slot)

    # -- parity access ----------------------------------------------------------------------------
    def debug(self, what):
        shapes = {DBG_RX: (np.float64, 64), DBG_RXVEC: (np.float64, 8), DBG_COEFFS: (np.float32, 8),
                  DBG_SCALARS: (np.float64, 8), DBG_PHASES: (np.float64, 8)}
        dt, n = shapes[what]
        out = np.zeros(n, dt)
        self._check(lib().wm_debug_get(self._h, what, out.ctypes.data))
        return out.reshape(8, 8) if what == DBG_RX else out

    def debug_set_coeffs(self, coeffs):
        if coeffs is None:
            self._check(lib().wm_debug_set_coeffs(self._h, None))
        else:
            c = np.ascontiguousarray(coeffs, np.float32)
            self._check(lib().wm_debug_set_coeffs(self._h, c.ctypes.data_as(C.POINTER(C.c_float))))

    def debug_plane(self, image, what):
        """e = I - pred (DBG_ERRSEQ) or the NVF mask (DBG_MASK_NVF) of a DeviceArray -> numpy (rows, cols)."""
        dst = DeviceArray(self, image.rows, image.cols, image.layout, F32, 1)
        d = image.desc()
        self._check(lib().wm_debug_plane(self._h, C.byref(d), what, dst.ptr))
        r = dst.numpy()
        dst.free()
        return r

    def debug_detect_planes(self, image, mask_type):
        """The detector's own kernel on an f32 DeviceArray, writing the planes it never materialises: -> (u, e_u, corr) as numpy."""
        du = DeviceArray(self, image.rows, image.cols, image.layout, F32, 1)
        de = DeviceArray(self, image.rows, image.cols, image.layout, F32, 1)
        corr = C.c_float(0.0)
        d = image.desc()
        self._check(lib().wm_debug_detect_planes(self._h, C.byref(d), mask_type, du.ptr, de.ptr, C.byref(corr)))
        u, eu = du.numpy(), de.numpy()
        du.free()
        de.free()
        return u, eu, corr.value

    def kernel_times(self, reset=True):
        """{name: (launches, total_ms)} accumulated while OPT_KERNEL_TIMING is on."""
        out = {}
        for k, name in enumerate(KERNEL_NAMES):
            ms = C.c_double(0.0)
            n = lib().wm_get_kernel_times(self._h, k, C.byref(ms), int(reset))
            out[name] = (int(n), ms.value)
        return out

    @property
    def launch_count(self):
        return int(lib().wm_launch_count(self._h))


class VideoProcessingContext:
    """videoprocessingcontext.hpp:13-29 minus the ffmpeg handles: frames come from memory.

    layout 0 (Y planes), a packed colour layout (PACKED_RGB / BGR / RGBA / BGRA: e.g. the BGR frames of cv2.VideoCapture) or a packed
    4:2:2 layout (PACKED_YUYV / UYVY: e.g. a V4L2 webcam's YUYV) or a 10-bit luma layout (Y10 / Y10_MSB: the Y plane of yuv420p10le or
    P010) or PACKED_V210 (e.g. a DeckLink's 10-bit YUV); linesize is the row pitch in bytes (default: dense rows of
    PACKED_BYTES[layout] * width bytes, v210_pitch(width) for v210)."""

    def __init__(self, watermark, height, width, watermark_interval, linesize=0, frame_stride=0, frames_on_device=False, layout=0):
        self.watermarkObj, self.height, self.width = watermark, height, width
        self.watermarkInterval = watermark_interval
        self.layout = layout
        self._c = wm_video_ctx(watermark._h, height, width, watermark_interval, linesize or (v210_pitch(width) if layout == PACKED_V210 else PACKED_BYTES.get(layout, 1) * width),
                               frame_stride, int(frames_on_device), layout)


def process_frames(ctx, mode, frames_ptr, out_ptr, first_index, n_frames, scalars):
    """main.cpp:319-410: per-frame embed (ME, u8 -> u8) or detect with interval gating on the global index."""
    n = lib().wm_process_frames(C.byref(ctx._c), mode, frames_ptr, out_ptr, first_index, n_frames,
                                scalars.ctypes.data_as(C.POINTER(C.c_float)))
    if n < 0:
        raise WatermarkError(int(n), lib().wm_last_error(ctx.watermarkObj._h).decode())
    return int(n)


def shard_frames(n_frames, rank, world):
    """Contiguous chunk of the global frame index owned by `rank` (SURVEY.md §8e): [first, first+count) — the library's own
    split (wm_shard_frames), so that every host language cuts the index range the same way."""
    first, count = C.c_int64(0), C.c_int64(0)
    lib().wm_shard_frames(n_frames, rank, world, C.byref(first), C.byref(count))
    return int(first.value), int(count.value)


def process_frames_multi(ctxs, mode, chunk_frames, chunk_out, first_index, n_frames, scalars):
    """wm_process_frames_multi: ctxs[g] (VideoProcessingContext, one per device / host thread) handles the g-th contiguous chunk of
    [first_index, first_index + n_frames); chunk_frames[g] / chunk_out[g] are raw pointers to the first frame of chunk g."""
    n = len(ctxs)
    arr = (C.POINTER(wm_video_ctx) * n)(*[C.pointer(c._c) for c in ctxs])
    fr = (C.c_void_p * n)(*[C.c_void_p(p) for p in chunk_frames])
    ou = (C.c_void_p * n)(*[C.c_void_p(p) for p in chunk_out]) if chunk_out is not None else None
    r = lib().wm_process_frames_multi(arr, n, mode, fr, ou, first_index, n_frames,
                                      scalars.ctypes.data_as(C.POINTER(C.c_float)) if scalars is not None else None)
    if r < 0:
        msgs = [lib().wm_last_error(c.watermarkObj._h).decode() for c in ctxs]
        raise WatermarkError(int(r), "; ".join(m for m in msgs if m))
    return int(r)
