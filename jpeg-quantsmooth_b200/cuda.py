"""ctypes binding of the C ABI in include/jpegqs_cuda.h (csrc/libjpegqs_b200.so) and the
Python mirror of the reference's public call for this path:

    ret, out = do_quantsmooth(image, flags, niter)      # reference libjpegqs.h:47-48

`image` is the flat equivalent of (j_decompress_ptr, coef_arrays) - see image.py.
There is no CPU fallback: a missing library or device raises QsError.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

from .image import CoefImage, JCS_YCbCr

_HERE = os.path.dirname(os.path.abspath(__file__))
MAX_COMP = 10


class QsError(RuntimeError):
    pass


def lib_path() -> str:
    # JPEGQS_B200_LIB: measurement builds of the same library (csrc/Makefile `experiments`,
    # `phase`) for tools/; never another implementation - there is no fallback of any kind
    return os.environ.get("JPEGQS_B200_LIB") or os.path.join(_HERE, "csrc", "libjpegqs_b200.so")


class _Comp(C.Structure):
    _fields_ = [("coef", C.c_void_p), ("wblk", C.c_uint32), ("hblk", C.c_uint32),
                ("h_samp", C.c_int32), ("v_samp", C.c_int32), ("has_qtbl", C.c_int32),
                ("quant", C.c_uint16 * 64), ("coef_up", C.c_void_p),
                ("rows", C.c_void_p), ("rows_up", C.c_void_p)]


class _Image(C.Structure):
    _fields_ = [("ncomp", C.c_int32), ("is_ycbcr", C.c_int32),
                ("image_width", C.c_uint32), ("image_height", C.c_uint32),
                ("comp", _Comp * MAX_COMP), ("upsampled", C.c_int32)]


class _Slab(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32),
                ("row0", C.c_uint32 * MAX_COMP), ("hblk_total", C.c_uint32 * MAX_COMP)]


PROGRESS_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int)

_lib = None


def load():
    """Load the CUDA extension; raises QsError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise QsError(f"{p} not built - run `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(there is no CPU fallback)")
    lib = C.CDLL(p)
    lib.jpegqs_cuda_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.jpegqs_cuda_destroy.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_last_error.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_last_error.restype = C.c_char_p
    lib.jpegqs_cuda_device_name.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_device_name.restype = C.c_char_p
    lib.jpegqs_cuda_last_device_ms.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_last_device_ms.restype = C.c_float
    lib.jpegqs_cuda_last_launches.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_host_alloc.argtypes = [C.c_size_t]
    lib.jpegqs_cuda_host_alloc.restype = C.c_void_p
    lib.jpegqs_cuda_host_free.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_run_host.argtypes = [C.c_void_p, C.POINTER(_Image), C.c_int, C.c_int, C.c_int,
                                         C.c_void_p, C.c_void_p]
    lib.jpegqs_cuda_run_device.argtypes = [C.c_void_p, C.POINTER(_Image), C.c_int, C.c_int, C.c_int,
                                           C.c_void_p, C.c_void_p, C.c_void_p]
    lib.jpegqs_cuda_run_batch.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Image), C.c_int, C.c_int,
                                          C.c_int, C.POINTER(C.c_int), C.c_void_p]
    lib.jpegqs_cuda_plane_bytes.argtypes = [C.c_uint32, C.c_uint32]
    lib.jpegqs_cuda_plane_bytes.restype = C.c_size_t
    lib.jpegqs_cuda_plane_stride.argtypes = [C.c_uint32]
    lib.jpegqs_cuda_render_rgb.argtypes = [C.c_void_p, C.POINTER(_Image), C.c_int, C.c_void_p, C.c_void_p]
    lib.jpegqs_cuda_set_profiling.argtypes = [C.c_void_p, C.c_int]
    lib.jpegqs_cuda_kernel_stats.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int),
                                             C.POINTER(C.c_float), C.POINTER(C.c_int)]
    lib.jpegqs_cuda_set_tuning.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.jpegqs_cuda_link_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.POINTER(C.c_void_p)]
    lib.jpegqs_cuda_link_destroy.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_link_export.argtypes = [C.c_void_p, C.c_void_p]
    lib.jpegqs_cuda_link_connect_ipc.argtypes = [C.c_void_p, C.c_void_p]
    lib.jpegqs_cuda_link_connect_local.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    lib.jpegqs_cuda_run_slab.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(_Image), C.POINTER(_Slab), C.c_int,
                                         C.c_int, C.c_int, C.c_void_p]
    lib.jpegqs_cuda_multi_create.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]
    lib.jpegqs_cuda_multi_destroy.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_multi_devices.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_multi_ctx.argtypes = [C.c_void_p, C.c_int]
    lib.jpegqs_cuda_multi_ctx.restype = C.c_void_p
    lib.jpegqs_cuda_multi_last_error.argtypes = [C.c_void_p]
    lib.jpegqs_cuda_multi_last_error.restype = C.c_char_p
    lib.jpegqs_cuda_multi_plan.argtypes = [C.c_void_p, C.POINTER(_Image)]
    lib.jpegqs_cuda_run_host_multi.argtypes = [C.c_void_p, C.POINTER(_Image), C.c_int, C.c_int]
    lib.jpegqs_cuda_tables.argtypes = [C.c_int, C.c_void_p]
    lib.jpegqs_cuda_orig_coef.argtypes = [C.c_int, C.c_int]
    _lib = lib
    return lib


def tables(flags: int) -> np.ndarray:
    """The weight tables the device uses (un-scaled), [64, 160|272] float32.  Host-only."""
    size = 272 if flags & 1 else 160
    out = np.zeros((64, size), dtype=np.float32)
    load().jpegqs_cuda_tables(flags, out.ctypes.data)
    return out


def orig_coef(coef: int, q: int) -> int:
    return load().jpegqs_cuda_orig_coef(coef, q)


def chunk_schedule(quant, max_coefs: int = 4, uniform: bool = True, merge: bool = True):
    """The smoothing kernel's chunk schedule for a quant table (or the table-independent one
    for quant=None): list of (type, first, [natural-order coefficient indices]).  Host-only."""
    lib = load()
    lib.jpegqs_cuda_chunk_schedule.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    out = np.zeros((64, 12), dtype=np.uint8)
    qp = None
    if quant is not None:
        qa = np.ascontiguousarray(quant, dtype=np.uint16).reshape(64)
        qp = qa.ctypes.data
    n = lib.jpegqs_cuda_chunk_schedule(qp, max_coefs, int(uniform) | (2 if merge else 0), out.ctypes.data)
    if n < 0:
        raise QsError(f"jpegqs_cuda_chunk_schedule: {n}")
    # type 3 ("mixed"): n full coefficients followed by the row-0 and the column-0 coefficient
    return [(int(r[0]), int(r[2]), [int(x) for x in r[4:4 + r[1] + (2 if r[0] == 3 else 0)]]) for r in out[:n]]


class PinnedArray:
    """int16 numpy view over pinned host memory from jpegqs_cuda_host_alloc."""

    def __init__(self, shape):
        n = int(np.prod(shape)) * 2
        self._lib = load()
        self._p = self._lib.jpegqs_cuda_host_alloc(max(n, 1))
        if not self._p:
            raise QsError("cudaMallocHost failed")
        buf = (C.c_int16 * (n // 2)).from_address(self._p)
        self.array = np.frombuffer(buf, dtype=np.int16).reshape(shape)

    def close(self):
        if self._p:
            self.array = None
            self._lib.jpegqs_cuda_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _fill_image(ci: _Image, image: CoefImage, coef_ptrs: Sequence[int], up_ptrs: Sequence[Optional[int]]):
    ci.ncomp = len(image.comps)
    ci.is_ycbcr = int(image.colorspace == JCS_YCbCr)
    ci.image_width, ci.image_height = image.width, image.height
    for i, c in enumerate(image.comps):
        cc = ci.comp[i]
        cc.coef = coef_ptrs[i]
        cc.wblk, cc.hblk, cc.h_samp, cc.v_samp = c.wblk, c.hblk, c.h_samp, c.v_samp
        cc.has_qtbl = int(c.quant is not None)
        if c.quant is not None:
            for k in range(64):
                cc.quant[k] = int(c.quant[k])
        cc.coef_up = up_ptrs[i] if i < len(up_ptrs) and up_ptrs[i] else None


class QsContext:
    """One device context (stream, tables, scratch arena).  Mirrors the process-wide state
    the reference keeps implicitly (its tables are rebuilt per call, quantsmooth.h:2460-2464)."""

    def __init__(self, device: int = -1):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.jpegqs_cuda_create(device, C.byref(h))
        if rc:
            raise QsError(f"jpegqs_cuda_create failed ({rc}): "
                          f"{self.lib.jpegqs_cuda_last_error(None).decode()}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.jpegqs_cuda_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise QsError(f"CUDA back end error {rc}: {self.lib.jpegqs_cuda_last_error(self.h).decode()}")
        return rc

    @property
    def device_name(self) -> str:
        return self.lib.jpegqs_cuda_device_name(self.h).decode()

    @property
    def last_device_ms(self) -> float:
        return float(self.lib.jpegqs_cuda_last_device_ms(self.h))

    @property
    def last_launches(self) -> int:
        return int(self.lib.jpegqs_cuda_last_launches(self.h))

    def set_profiling(self, on: bool):
        self.lib.jpegqs_cuda_set_profiling(self.h, int(on))

    def set_tuning(self, key: int, value: int):
        self._check(self.lib.jpegqs_cuda_set_tuning(self.h, key, value))

    def kernel_stats(self):
        """(idct_ms, idct_launches, smooth_ms, smooth_launches) of the last run_* call."""
        a, b, c, d = C.c_float(), C.c_int(), C.c_float(), C.c_int()
        self.lib.jpegqs_cuda_kernel_stats(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
        return a.value, b.value, c.value, d.value

    # ---- whole image, host buffers (the call a user of the reference makes) ----
    def do_quantsmooth(self, image: CoefImage, flags: int, niter: int, progprec: int = 0,
                       progress=None, inplace: bool = False, pinned: bool = False):
        """pinned=True stages the coefficient arrays in page-locked memory (what the C entry
        point do_quantsmooth does): only then the upload/download slab pipeline is used."""
        out = image if inplace else image.clone()
        keep = []
        ptrs, ups = [], []
        for c in out.comps:
            c.coef = np.ascontiguousarray(c.coef, dtype=np.int16)
            if pinned and c.coef.size:
                pa = PinnedArray(c.coef.shape)
                pa.array[...] = c.coef
                keep.append((pa, c))
                ptrs.append(pa.array.ctypes.data)
            else:
                ptrs.append(c.coef.ctypes.data)
        up_arrays = []
        if len(out.comps) >= 3:
            y = out.comps[0]
            ups.append(None)
            for _ in range(2):
                a = np.zeros((y.hblk, y.wblk, 64), dtype=np.int16)
                up_arrays.append(a)
                ups.append(a.ctypes.data)
        ci = _Image()
        _fill_image(ci, out, ptrs, ups)
        cb = None
        if progress is not None:
            cb = PROGRESS_FN(lambda d, cur, mx: int(progress(cur, mx)))
            keep.append(cb)
        ret = self._check(self.lib.jpegqs_cuda_run_host(
            self.h, C.byref(ci), flags & 0x7f, niter, progprec,
            C.cast(cb, C.c_void_p) if cb else None, None))
        for item in keep:
            if isinstance(item, tuple):
                pa, c = item
                c.coef[...] = pa.array
                pa.close()
        self._collect(out, ci, up_arrays)
        return ret, out

    @staticmethod
    def _collect(out: CoefImage, ci: _Image, up_arrays):
        for i, c in enumerate(out.comps):
            if ci.upsampled and i in (1, 2):
                c.coef = up_arrays[i - 1]
            if ci.upsampled:
                c.h_samp = c.v_samp = 1
            if c.quant is not None:
                c.quant = np.array(list(ci.comp[i].quant), dtype=np.uint16)

    def render_rgb(self, image: CoefImage) -> np.ndarray:
        """Decode a coefficient image (smoothed, or still quantized) to RGB [H, W, 3] uint8 the way
        libjpeg would (islow IDCT, fancy up-sampling, fixed-point YCbCr->RGB)."""
        ptrs = []
        keep = []
        for c in image.comps:
            a = np.ascontiguousarray(c.coef, dtype=np.int16)
            keep.append(a)
            ptrs.append(a.ctypes.data)
        ci = _Image()
        _fill_image(ci, image, ptrs, [])
        out = np.zeros((image.height, image.width, 3), dtype=np.uint8)
        self._check(self.lib.jpegqs_cuda_render_rgb(self.h, C.byref(ci), 0, out.ctypes.data, None))
        return out

    def run_batch_host(self, images: List[CoefImage], flags: int, niter: int):
        outs = [im.clone() for im in images]
        arr = (_Image * len(outs))()
        ups_all = []
        for n, out in enumerate(outs):
            ptrs, ups, up_arrays = [], [], []
            for c in out.comps:
                c.coef = np.ascontiguousarray(c.coef, dtype=np.int16)
                ptrs.append(c.coef.ctypes.data)
            if len(out.comps) >= 3:
                y = out.comps[0]
                ups.append(None)
                for _ in range(2):
                    a = np.zeros((y.hblk, y.wblk, 64), dtype=np.int16)
                    up_arrays.append(a)
                    ups.append(a.ctypes.data)
            _fill_image(arr[n], out, ptrs, ups)
            ups_all.append(up_arrays)
        rets = (C.c_int * len(outs))()
        self._check(self.lib.jpegqs_cuda_run_batch(self.h, len(outs), arr, flags & 0x7f, niter, 0, rets, None))
        for n, out in enumerate(outs):
            self._collect(out, arr[n], ups_all[n])
        return list(rets), outs

    # ---- device-resident buffers (torch tensors or raw pointers) ----
    def run_device(self, image: CoefImage, coef_ptrs: Sequence[int], up_ptrs: Sequence[Optional[int]],
                   flags: int, niter: int, stream: int = 0):
        """image carries geometry + quant tables; coef_ptrs/up_ptrs are device pointers.
        Returns (ret, upsampled)."""
        ci = _Image()
        _fill_image(ci, image, coef_ptrs, up_ptrs)
        ret = self._check(self.lib.jpegqs_cuda_run_device(self.h, C.byref(ci), flags & 0x7f, niter, 0,
                                                         None, None, C.c_void_p(stream or None)))
        return ret, bool(ci.upsampled)

    def run_batch_device(self, images: List[CoefImage], coef_ptrs: List[Sequence[int]],
                         up_ptrs: List[Sequence[Optional[int]]], flags: int, niter: int, stream: int = 0):
        arr = (_Image * len(images))()
        for n, im in enumerate(images):
            _fill_image(arr[n], im, coef_ptrs[n], up_ptrs[n] if up_ptrs else [])
        rets = (C.c_int * len(images))()
        self._check(self.lib.jpegqs_cuda_run_batch(self.h, len(images), arr, flags & 0x7f, niter, 1, rets,
                                                   C.c_void_p(stream or None)))
        return list(rets), [bool(a.upsampled) for a in arr]

    # ---- one slab of a sharded image (include/jpegqs_cuda.h "one image sharded by MCU rows") ----
    def run_slab(self, link, slab: CoefImage, rank: int, world: int, row0: Sequence[int],
                 hblk_total: Sequence[int], flags: int, niter: int, coef_ptrs=None, up_ptrs=None, stream: int = 0):
        """slab: CoefImage whose components hold this rank's block rows (width / height = the
        WHOLE image's).  Host arrays (coef_ptrs None: slab.comps[].coef, modified IN PLACE, results
        for UPSAMPLE_UV in the returned arrays) or device pointers (coef_ptrs / up_ptrs).
        Returns (ret, upsampled, up_arrays)."""
        on_device = coef_ptrs is not None
        up_arrays = []
        if not on_device:
            coef_ptrs, up_ptrs = [], []
            for c in slab.comps:
                c.coef = np.ascontiguousarray(c.coef, dtype=np.int16)
                coef_ptrs.append(c.coef.ctypes.data)
            if len(slab.comps) >= 3:
                y = slab.comps[0]
                up_ptrs.append(None)
                for _ in range(2):
                    a = np.zeros((y.hblk, y.wblk, 64), dtype=np.int16)
                    up_arrays.append(a)
                    up_ptrs.append(a.ctypes.data)
        ci = _Image()
        _fill_image(ci, slab, coef_ptrs, up_ptrs or [])
        g = _Slab()
        g.rank, g.world = rank, world
        for k in range(len(slab.comps)):
            g.row0[k], g.hblk_total[k] = int(row0[k]), int(hblk_total[k])
        ret = self._check(self.lib.jpegqs_cuda_run_slab(self.h, link.h if link is not None else None, C.byref(ci),
                                                       C.byref(g), flags & 0x7f, niter, int(on_device),
                                                       C.c_void_p(stream or None)))
        if not on_device:
            for i, c in enumerate(slab.comps):
                if c.quant is not None:
                    c.quant = np.array(list(ci.comp[i].quant), dtype=np.uint16)
        return ret, bool(ci.upsampled), up_arrays

    def plane_bytes(self, wblk, hblk) -> int:
        return int(self.lib.jpegqs_cuda_plane_bytes(wblk, hblk))

    def plane_stride(self, wblk) -> int:
        return int(self.lib.jpegqs_cuda_plane_stride(wblk))

    def plane_pad(self) -> int:
        return int(self.lib.jpegqs_cuda_plane_pad())


class QsLink:
    """This rank's mailbox + its view of the other ranks' (jpegqs_cuda_link)."""

    def __init__(self, ctx: QsContext, rank: int, world: int, max_wblk: int):
        self.ctx, self.lib, self.rank, self.world = ctx, ctx.lib, rank, world
        h = C.c_void_p()
        ctx._check(self.lib.jpegqs_cuda_link_create(ctx.h, rank, world, max_wblk, C.byref(h)))
        self.h = h

    def export(self) -> bytes:
        n = self.lib.jpegqs_cuda_link_handle_bytes()
        buf = C.create_string_buffer(n)
        self.ctx._check(self.lib.jpegqs_cuda_link_export(self.h, buf))
        return buf.raw

    def connect_ipc(self, handles: Sequence[bytes]):
        blob = b"".join(handles)
        self.ctx._check(self.lib.jpegqs_cuda_link_connect_ipc(self.h, blob))

    @staticmethod
    def connect_local(links: Sequence["QsLink"]):
        arr = (C.c_void_p * len(links))(*[l.h for l in links])
        links[0].ctx._check(links[0].lib.jpegqs_cuda_link_connect_local(arr, len(links)))

    def close(self):
        if getattr(self, "h", None):
            self.lib.jpegqs_cuda_link_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class QsMulti:
    """Several devices of this process behind one call (jpegqs_cuda_multi): what the C entry
    point do_quantsmooth uses when JPEGQS_GPUS is set."""

    def __init__(self, devices):
        self.lib = load()
        if isinstance(devices, int):
            n, arr = devices, None
        else:
            n, arr = len(devices), (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        rc = self.lib.jpegqs_cuda_multi_create(n, arr, C.byref(h))
        if rc:
            raise QsError(f"jpegqs_cuda_multi_create failed ({rc}): {self.lib.jpegqs_cuda_last_error(None).decode()}")
        self.h = h

    def _image(self, out: CoefImage):
        ptrs, ups, up_arrays = [], [], []
        for c in out.comps:
            c.coef = np.ascontiguousarray(c.coef, dtype=np.int16)
            ptrs.append(c.coef.ctypes.data)
        if len(out.comps) >= 3:
            y = out.comps[0]
            ups.append(None)
            for _ in range(2):
                a = np.zeros((y.hblk, y.wblk, 64), dtype=np.int16)
                up_arrays.append(a)
                ups.append(a.ctypes.data)
        ci = _Image()
        _fill_image(ci, out, ptrs, ups)
        return ci, up_arrays

    def plan(self, image: CoefImage) -> int:
        ci, _ = self._image(image.clone())
        return int(self.lib.jpegqs_cuda_multi_plan(self.h, C.byref(ci)))

    def do_quantsmooth(self, image: CoefImage, flags: int, niter: int):
        out = image.clone()
        ci, up_arrays = self._image(out)
        rc = self.lib.jpegqs_cuda_run_host_multi(self.h, C.byref(ci), flags & 0x7f, niter)
        if rc < 0:
            raise QsError(f"CUDA back end error {rc}: {self.lib.jpegqs_cuda_multi_last_error(self.h).decode()}")
        QsContext._collect(out, ci, up_arrays)
        return rc, out

    def close(self):
        if getattr(self, "h", None):
            self.lib.jpegqs_cuda_multi_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def default_context(device: int = -1) -> QsContext:
    if device not in _default_ctx:
        _default_ctx[device] = QsContext(device)
    return _default_ctx[device]


def do_quantsmooth(image: CoefImage, flags: int, niter: int, progprec: int = 0, progress=None,
                   device: int = -1):
    """Python mirror of `int do_quantsmooth(srcinfo, coef_arrays, opts)` (reference
    libjpegqs.h:47-48): returns (stop, smoothed image)."""
    return default_context(device).do_quantsmooth(image, flags, niter, progprec, progress)
