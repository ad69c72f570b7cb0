"""timg_b200 -- Python door onto libb200timg.so (the C ABI in include/b200timg.h).

This module is harness plumbing for tests and bench.py: it loads the in-tree shared
library with ctypes, declares every symbol of the ABI, and offers small numpy/torch
conveniences.  The product is the CUDA library; there is no Python or CPU fallback:
loading fails loudly if the library is missing, and Context() raises if no B200 is
visible.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200TIMG_LIBFILE") or os.path.join(_HERE, "libb200timg.so")   # tuning runs load a variant build

OK, EINVAL, ENOMEM, ECUDA, ENOSPC, ENODEV = 0, -1, -2, -3, -4, -5
QUARTER, UPPER, COLOR8, FAST_SCALE, BILINEAR_SCALE = 1, 2, 4, 8, 16
FMT_RGBA, FMT_RGB32, FMT_I420, FMT_NV12, FMT_FULL_RANGE = 0, 1, 2, 3, 0x10

u8p = C.POINTER(C.c_uint8)
u64p = C.POINTER(C.c_uint64)


class FitOpts(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("cell_x_px", C.c_int), ("cell_y_px", C.c_int),
                ("width_stretch", C.c_float), ("upscale", C.c_int), ("upscale_integer", C.c_int),
                ("fill_width", C.c_int), ("fill_height", C.c_int)]


class Batch(C.Structure):
    _fields_ = [("n_frames", C.c_int), ("src_w", C.c_int), ("src_h", C.c_int), ("src_fmt", C.c_int),
                ("out_w", C.c_int), ("out_h", C.c_int), ("has_bg", C.c_int), ("bg", C.c_uint32),
                ("pattern", C.c_uint32), ("pattern_w", C.c_int), ("pattern_h", C.c_int),
                ("flags", C.c_int), ("x_indent_cells", C.c_int), ("animation", C.c_int)]


# name -> (restype, argtypes); this table IS the list of exported symbols tests check.
ABI = {
    "b200timg_version": (C.c_int, []),
    "b200timg_ctx_create": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "b200timg_ctx_destroy": (None, [C.c_void_p]),
    "b200timg_last_error": (C.c_char_p, [C.c_void_p]),
    "b200timg_kernel_launches": (C.c_uint64, [C.c_void_p]),
    "b200timg_calc_fit": (C.c_int, [C.POINTER(FitOpts), C.c_int, C.c_int, C.c_int,
                                    C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "b200timg_as256": (C.c_int, [C.c_uint32]),
    "b200timg_scale_rgba": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, u8p, C.c_int, C.c_int]),
    "b200timg_scale_rgba_mode": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, u8p, C.c_int, C.c_int, C.c_int]),
    "b200timg_yuv_scale": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, u8p, C.c_int, C.c_int]),
    "b200timg_compose_bg": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint32,
                                      C.c_int, C.c_int, C.c_int]),
    "b200timg_compose_bg_resident": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint32,
                                               C.c_int, C.c_int, C.c_int]),
    "b200timg_has_transparency": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "b200timg_blocks_bound": (C.c_size_t, [C.c_int, C.c_int]),
    "b200timg_blocks_encode": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, u8p, C.c_int, C.c_int,
                                         C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "b200timg_sixel_bound": (C.c_size_t, [C.c_int, C.c_int]),
    "b200timg_sixel_encode": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_char_p, C.c_size_t,
                                        C.POINTER(C.c_size_t)]),
    "b200timg_blocks_batch_dev": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p, C.c_void_p, C.c_size_t,
                                            C.c_void_p]),
    "b200timg_sixel_batch_dev": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p, C.c_void_p, C.c_size_t,
                                           C.c_void_p]),
    "b200timg_blocks_batch": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.c_void_p]),
    "b200timg_sixel_batch": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p, C.c_void_p, C.c_size_t,
                                       C.c_void_p]),
    "b200timg_scale_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                     C.c_int, C.c_int]),
    "b200timg_compose_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32,
                                       C.c_uint32, C.c_int, C.c_int, C.c_int]),
    "b200timg_sixel_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t,
                                     C.c_void_p]),
    "b200timg_exif_op": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p]),
    "b200timg_exif_op_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "b200timg_trim_bbox": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "b200timg_windows": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_longlong, C.c_int,
                                   C.c_int, C.c_longlong, C.c_int, u8p]),
    "b200timg_windows_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_longlong,
                                       C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p]),
    "b200timg_png_size": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "b200timg_base64_size": (C.c_size_t, [C.c_size_t]),
    "b200timg_png_encode": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, u8p, C.c_size_t, C.c_char_p, C.c_size_t]),
    "b200timg_png_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "b200timg_png_bound": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "b200timg_png_encode_level": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p, C.c_size_t,
                                            C.POINTER(C.c_size_t), C.c_char_p, C.c_size_t]),
    "b200timg_png_batch_level_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                               C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200timg_gather_unique_id": (C.c_int, [C.c_char_p]),
    "b200timg_gather_init": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_int]),
    "b200timg_gather_attach": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "b200timg_gather_shutdown": (None, [C.c_void_p]),
    "b200timg_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_int]),
    "b200timg_gather_wait": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "b200timg_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "b200timg_profile_report": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t]),
    "b200timg_sixel_debug": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200timg_resample_plan": (C.c_int, [C.c_int] * 5 + [C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p,
                                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
}

_lib = None


def build(verbose=False):
    """Compile every CUDA source for sm_100a into timg_b200/libb200timg.so (in-tree)."""
    subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"], check=True,
                   stdout=None if verbose else subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(timg_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in ABI.items():
            f = getattr(L, name)          # AttributeError if a declared symbol is not exported
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


class B200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"b200timg error {code}: {msg}")
        self.code = code


def rgba_u32(r, g, b, a=255):
    return (r & 255) | ((g & 255) << 8) | ((b & 255) << 16) | ((a & 255) << 24)


def calc_fit(iw, ih, width, height, cell_x=1, cell_y=2, stretch=1.0, upscale=False,
             upscale_integer=False, fill_width=False, fill_height=False, rotated=False):
    o = FitOpts(width, height, cell_x, cell_y, stretch, int(upscale), int(upscale_integer),
                int(fill_width), int(fill_height))
    tw, th = C.c_int(), C.c_int()
    r = lib().b200timg_calc_fit(C.byref(o), iw, ih, int(rotated), C.byref(tw), C.byref(th))
    if r < 0:
        raise B200Error(r, "calc_fit")
    return bool(r), tw.value, th.value


def resample_plan(iw, ih, ow, oh, axis):
    """Host-side resampling plan of one axis as numpy arrays (see include/b200timg.h)."""
    n = ow if axis == 0 else oh
    widest, flags = C.c_int(), C.c_int()
    rc = lib().b200timg_resample_plan(iw, ih, ow, oh, axis, C.byref(widest), C.byref(flags), None, None, None,
                                      None, 1 << 62)
    if rc != OK:
        raise B200Error(rc, "resample_plan")
    first, count, lead = (np.zeros(n, np.int32) for _ in range(3))
    coeff = np.zeros(n * widest.value, np.float32)
    rc = lib().b200timg_resample_plan(iw, ih, ow, oh, axis, None, None, first.ctypes.data, count.ctypes.data,
                                      lead.ctypes.data, coeff.ctypes.data, coeff.size)
    if rc != OK:
        raise B200Error(rc, "resample_plan")
    return dict(widest=widest.value, flags=flags.value, first=first, count=count, lead=lead,
                coeff=coeff.reshape(n, widest.value))


def _np_ptr(a):
    return a.ctypes.data_as(u8p)


class Context:
    """One b200timg_ctx.  Raises B200Error(ENODEV) when no CUDA device is usable."""

    def __init__(self, device=0, stream=None):
        h = C.c_void_p()
        rc = lib().b200timg_ctx_create(device, stream, C.byref(h))
        if rc != OK:
            raise B200Error(rc, "ctx_create failed (no usable CUDA device? this library has no CPU path)")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None) and _lib is not None:
            _lib.b200timg_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def _chk(self, rc):
        if rc != OK:
            raise B200Error(rc, lib().b200timg_last_error(self.h).decode())

    @property
    def launches(self):
        return lib().b200timg_kernel_launches(self.h)

    # ---- single-frame host entry points (numpy in / numpy or bytes out)
    def scale(self, img, ow, oh, fmt=FMT_RGBA, fast=False):
        """fast: False/0 bit-exact STB semantics, True/1 <= 1 LSB mode, 2 libswscale-style bilinear."""
        img = np.ascontiguousarray(img, dtype=np.uint8)
        ih, iw = img.shape[:2]
        out = np.empty((oh, ow, 4), np.uint8)
        self._chk(lib().b200timg_scale_rgba_mode(self.h, _np_ptr(img), iw, ih, fmt, _np_ptr(out), ow, oh, int(fast)))
        return out

    def yuv_scale(self, yuv, iw, ih, ow, oh, fmt=FMT_I420):
        """yuv: flat uint8 array of iw*ih*3/2 bytes (I420 or NV12) -> RGBA [oh, ow, 4]."""
        yuv = np.ascontiguousarray(yuv, dtype=np.uint8).reshape(-1)
        assert yuv.size == iw * ih * 3 // 2
        out = np.empty((oh, ow, 4), np.uint8)
        self._chk(lib().b200timg_yuv_scale(self.h, _np_ptr(yuv), iw, ih, fmt, _np_ptr(out), ow, oh))
        return out

    def exif_op(self, fb, mirror=False, angle=0):
        fb = np.ascontiguousarray(fb, dtype=np.uint8)
        h, w = fb.shape[:2]
        out = np.empty((w, h, 4) if angle in (90, -90) else (h, w, 4), np.uint8)
        self._chk(lib().b200timg_exif_op(self.h, _np_ptr(fb), w, h, int(mirror), angle, _np_ptr(out)))
        return out

    def trim_bbox(self, fb):
        fb = np.ascontiguousarray(fb, dtype=np.uint8)
        h, w = fb.shape[:2]
        r = (C.c_int * 4)()
        self._chk(lib().b200timg_trim_bbox(self.h, _np_ptr(fb), w, h, r))
        return tuple(r)

    def windows(self, img, dw, dh, x0=0, y0=0, dx=0, dy=0, first_pos=0, n_pos=1):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        h, w = img.shape[:2]
        out = np.empty((n_pos, dh, dw, 4), np.uint8)
        self._chk(lib().b200timg_windows(self.h, _np_ptr(img), w, h, dw, dh, x0, y0, dx, dy, first_pos, n_pos, _np_ptr(out)))
        return out

    def png_encode(self, fb, rgb24=False, want_base64=True, level=0):
        """(PNG bytes, base64 text or None) of an RGBA frame, as the kitty / iTerm2 canvases would send it.
        level: timg's --compress (0 stored blocks, 1..9 deflate-compressed)."""
        fb = np.ascontiguousarray(fb, dtype=np.uint8)
        h, w = fb.shape[:2]
        if level == 0:
            n = lib().b200timg_png_size(w, h, int(rgb24))
            out = np.empty(n, np.uint8)
            nb = lib().b200timg_base64_size(n)
            b64 = C.create_string_buffer(nb) if want_base64 else None
            self._chk(lib().b200timg_png_encode(self.h, _np_ptr(fb), w, h, int(rgb24), _np_ptr(out), n, b64, nb if want_base64 else 0))
            return out.tobytes(), (b64.raw if want_base64 else None)
        cap = lib().b200timg_png_bound(w, h, int(rgb24), level)
        out = np.empty(cap, np.uint8)
        nb = lib().b200timg_base64_size(cap)
        b64 = C.create_string_buffer(nb) if want_base64 else None
        n = C.c_size_t()
        self._chk(lib().b200timg_png_encode_level(self.h, _np_ptr(fb), w, h, int(rgb24), level, _np_ptr(out), cap, C.byref(n),
                                                  b64, nb if want_base64 else 0))
        data = out[:n.value].tobytes()
        return data, (b64.raw[:lib().b200timg_base64_size(n.value)] if want_base64 else None)

    def compose_bg(self, fb, bg, pattern=0, pw=0, ph=0, start_row=0, has_bg=True):
        out = np.ascontiguousarray(fb, dtype=np.uint8).copy()
        h, w = out.shape[:2]
        self._chk(lib().b200timg_compose_bg(self.h, _np_ptr(out), w, h, int(has_bg), bg, pattern, pw, ph,
                                            start_row))
        return out

    def has_transparency(self, fb, start_row=0):
        fb = np.ascontiguousarray(fb, dtype=np.uint8)
        h, w = fb.shape[:2]
        r = C.c_int()
        self._chk(lib().b200timg_has_transparency(self.h, _np_ptr(fb), w, h, start_row, C.byref(r)))
        return bool(r.value)

    def blocks_encode(self, fb, prev=None, flags=0, x_indent_cells=0):
        fb = np.ascontiguousarray(fb, dtype=np.uint8)
        h, w = fb.shape[:2]
        cap = lib().b200timg_blocks_bound(w, h) + 64
        buf = C.create_string_buffer(cap)
        n = C.c_size_t()
        pp = None
        if prev is not None:
            prev = np.ascontiguousarray(prev, dtype=np.uint8)
            assert prev.shape == fb.shape
            pp = _np_ptr(prev)
        self._chk(lib().b200timg_blocks_encode(self.h, _np_ptr(fb), w, h, pp, flags, x_indent_cells, buf, cap,
                                               C.byref(n)))
        return buf.raw[:n.value]

    def sixel_encode(self, fb):
        fb = np.ascontiguousarray(fb, dtype=np.uint8)
        h, w = fb.shape[:2]
        cap = 4096 + 6 * w * h
        buf = C.create_string_buffer(cap)
        n = C.c_size_t()
        rc = lib().b200timg_sixel_encode(self.h, _np_ptr(fb), w, h, buf, cap, C.byref(n))
        if rc == ENOSPC:                       # sized exactly by the library before anything is written
            cap = n.value
            buf = C.create_string_buffer(cap)
            rc = lib().b200timg_sixel_encode(self.h, _np_ptr(fb), w, h, buf, cap, C.byref(n))
        self._chk(rc)
        return buf.raw[:n.value]

    def profile(self, enable=True):
        self._chk(lib().b200timg_profile(self.h, int(enable)))

    def profile_report(self):
        """{kernel name: (launches, total_ms)} since profile(True)."""
        buf = C.create_string_buffer(1 << 16)
        self._chk(lib().b200timg_profile_report(self.h, buf, len(buf)))
        out = {}
        for line in buf.value.decode().splitlines():
            name, n, ms = line.split()
            out[name] = (int(n), float(ms))
        return out

    def sixel_debug(self, w, h):
        """(palette[n,3] uint8, origcolors, index[h,w]) of the last sixel_encode call."""
        pal = np.zeros(256, np.uint32)
        cnt = np.zeros(2, np.uint32)
        idx = np.zeros((h, w), np.uint8)
        self._chk(lib().b200timg_sixel_debug(self.h, pal.ctypes.data, cnt.ctypes.data, idx.ctypes.data, idx.size))
        rgb = np.stack([pal & 255, (pal >> 8) & 255, (pal >> 16) & 255], -1).astype(np.uint8)
        return rgb[: int(cnt[0])], int(cnt[1]), idx

    # ---- batches, host buffers (numpy [n,h,w,4]) -> list of bytes
    def _batch_host(self, fn, frames, b, sixel=False):
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        n = frames.shape[0]
        if sixel:
            cap = n * (4096 + 6 * b.out_w * (b.out_h + 5))      # far above typical (~1 B/px); ENOSPC reports the need
        else:
            cap = lib().b200timg_blocks_bound(b.out_w, b.out_h) * n + 64
        out = np.empty(cap, np.uint8)
        offs = np.zeros(n + 1, np.uint64)
        self._chk(fn(self.h, C.byref(b), frames.ctypes.data, out.ctypes.data, cap, offs.ctypes.data))
        return [out[int(offs[i]):int(offs[i + 1])].tobytes() for i in range(n)]

    def blocks_batch(self, frames, b):
        return self._batch_host(lib().b200timg_blocks_batch, frames, b)

    def sixel_batch(self, frames, b):
        return self._batch_host(lib().b200timg_sixel_batch, frames, b, sixel=True)
