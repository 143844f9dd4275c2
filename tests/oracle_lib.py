"""ctypes bindings for the TEST INFRASTRUCTURE under oracle/:
  - oracle/_ref/libqsref_{scalar,avx512}.so : the unmodified reference (built by build() through
    oracle/Makefile where the reference's sources are present)
  - oracle/libqs_oracle.so                  : the C restatement
  - oracle/libfakejpeg.so                   : fake libjpeg front end used to drive any
    do_quantsmooth-shaped function through the libjpeg-facing boundary.
Nothing in the product imports this module."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE, "_ref")


def ensure_built():
    need = [os.path.join(ORACLE, "libqs_oracle.so"), os.path.join(ORACLE, "libfakejpeg.so")]
    src = [os.path.join(ORACLE, "qs_oracle.c"), os.path.join(ORACLE, "fakejpeg.c")]
    stale = any((not os.path.exists(n)) or os.path.getmtime(n) < os.path.getmtime(s)
                for n, s in zip(need, src))
    if stale:
        subprocess.run(["make", "-C", ORACLE, "restatement", "fake"], check=True, capture_output=True)


def have_ref(variant="scalar"):
    return os.path.exists(os.path.join(REF_DIR, f"libqsref_{variant}.so"))


class Control(C.Structure):          # jpegqs_control_t, include/libjpegqs.h
    _fields_ = [("flags", C.c_int), ("niter", C.c_int), ("threads", C.c_int),
                ("progprec", C.c_int), ("userdata", C.c_void_p), ("progress", C.c_void_p)]


PROGRESS_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int)


class FakeImage(C.Structure):        # fake_image, oracle/fakejpeg.c
    _fields_ = [("num_components", C.c_int), ("color_space", C.c_int),
                ("image_width", C.c_uint), ("image_height", C.c_uint),
                ("h_samp", C.c_int * 4), ("v_samp", C.c_int * 4), ("quant_tbl_no", C.c_int * 4),
                ("width_in_blocks", C.c_uint * 4), ("height_in_blocks", C.c_uint * 4),
                ("quant", (C.c_uint16 * 64) * 4), ("slot_present", C.c_int),
                ("coef", C.c_void_p * 4), ("coef_up", C.c_void_p * 2),
                ("upsampled", C.c_int), ("max_h_samp", C.c_int), ("max_v_samp", C.c_int),
                ("scatter_rows", C.c_int)]


_cache = {}


def _load(path):
    if path not in _cache:
        _cache[path] = C.CDLL(path)
    return _cache[path]


def fakejpeg():
    return _load(os.path.join(ORACLE, "libfakejpeg.so"))


def reflib(variant="scalar"):
    lib = _load(os.path.join(REF_DIR, f"libqsref_{variant}.so"))
    lib.qsref_variant.restype = C.c_char_p
    lib.qsref_take_log.restype = C.c_char_p
    return lib


def oraclelib():
    lib = _load(os.path.join(ORACLE, "libqs_oracle.so"))
    lib.qso_orig_coef.restype = C.c_int
    return lib


def run_libjpeg_boundary(fn_ptr, image, flags, niter, threads=0, progprec=0, progress=None,
                         scatter_rows=False):
    """Drive a `int fn(j_decompress_ptr, jvirt_barray_ptr*, jpegqs_control_t*)` through the
    fake libjpeg front end.  Returns (ret, result_image)."""
    from jpegqs_b200.image import CoefImage, Component
    out = image.clone()
    fi = FakeImage()
    fi.num_components = len(out.comps)
    fi.color_space = out.colorspace
    fi.image_width, fi.image_height = out.width, out.height
    fi.scatter_rows = int(scatter_rows)
    keep = []
    slots = 0
    for i, c in enumerate(out.comps):
        fi.h_samp[i], fi.v_samp[i], fi.quant_tbl_no[i] = c.h_samp, c.v_samp, c.quant_tbl_no
        fi.width_in_blocks[i], fi.height_in_blocks[i] = c.wblk, c.hblk
        c.coef = np.ascontiguousarray(c.coef, dtype=np.int16)
        fi.coef[i] = c.coef.ctypes.data
        if c.quant is not None:
            slots |= 1 << c.quant_tbl_no
            for k in range(64):
                fi.quant[c.quant_tbl_no][k] = int(c.quant[k])
    fi.slot_present = slots
    ups = []
    if len(out.comps) >= 3:
        y = out.comps[0]
        for j in range(2):
            a = np.zeros((y.hblk, y.wblk, 64), dtype=np.int16)
            ups.append(a)
            fi.coef_up[j] = a.ctypes.data
    ctl = Control(flags=flags, niter=niter, threads=threads, progprec=progprec)
    if progress is not None:
        cb = PROGRESS_FN(progress)
        keep.append(cb)
        ctl.progress = C.cast(cb, C.c_void_p)
    f = fakejpeg().fakejpeg_call
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.POINTER(FakeImage), C.POINTER(Control)]
    ret = f(C.cast(fn_ptr, C.c_void_p), C.byref(fi), C.byref(ctl))
    for i, c in enumerate(out.comps):
        if fi.upsampled and i in (1, 2):
            c.coef = ups[i - 1]
        c.h_samp, c.v_samp = fi.h_samp[i], fi.v_samp[i]
        assert (c.wblk, c.hblk) == (fi.width_in_blocks[i], fi.height_in_blocks[i])
        if c.quant is not None:
            c.quant = np.array(list(fi.quant[c.quant_tbl_no]), dtype=np.uint16)
    return ret, out


class BoundarySession:
    """A live fake `j_decompress_ptr` + coefficient arrays (oracle/fakejpeg.c session API):
    `run(fn_ptr, flags, niter)` calls fn(&cinfo, coef_arrays, &opts) and nothing else, so a
    benchmark can time exactly the drop-in call; `load()` restores the input, `result()` copies
    the arrays out.  scatter_rows: every block row separately malloc'd (pageable, non-adjacent),
    which is how libjpeg's memory manager hands rows over."""

    def __init__(self, image, scatter_rows=True):
        self.image = image.clone()
        self.fi = fi = FakeImage()
        out = self.image
        fi.num_components = len(out.comps)
        fi.color_space = out.colorspace
        fi.image_width, fi.image_height = out.width, out.height
        fi.scatter_rows = int(scatter_rows)
        slots = 0
        for i, c in enumerate(out.comps):
            fi.h_samp[i], fi.v_samp[i], fi.quant_tbl_no[i] = c.h_samp, c.v_samp, c.quant_tbl_no
            fi.width_in_blocks[i], fi.height_in_blocks[i] = c.wblk, c.hblk
            c.coef = np.ascontiguousarray(c.coef, dtype=np.int16)
            fi.coef[i] = c.coef.ctypes.data
            if c.quant is not None:
                slots |= 1 << c.quant_tbl_no
                for k in range(64):
                    fi.quant[c.quant_tbl_no][k] = int(c.quant[k])
        fi.slot_present = slots
        self.ups = []
        if len(out.comps) >= 3:
            y = out.comps[0]
            for j in range(2):
                a = np.zeros((y.hblk, y.wblk, 64), dtype=np.int16)
                self.ups.append(a)
                fi.coef_up[j] = a.ctypes.data
        lib = fakejpeg()
        lib.fakejpeg_open.restype = C.c_void_p
        lib.fakejpeg_open.argtypes = [C.POINTER(FakeImage)]
        lib.fakejpeg_load.argtypes = [C.c_void_p, C.POINTER(FakeImage)]
        lib.fakejpeg_run.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Control)]
        lib.fakejpeg_run.restype = C.c_int
        lib.fakejpeg_store.argtypes = [C.c_void_p, C.POINTER(FakeImage)]
        lib.fakejpeg_close.argtypes = [C.c_void_p]
        self.lib = lib
        self.h = lib.fakejpeg_open(C.byref(fi))

    def load(self):
        self.lib.fakejpeg_load(self.h, C.byref(self.fi))

    def run(self, fn_ptr, flags, niter, threads=0):
        ctl = Control(flags=flags, niter=niter, threads=threads, progprec=0)
        return self.lib.fakejpeg_run(self.h, C.cast(fn_ptr, C.c_void_p), C.byref(ctl))

    def result(self):
        """Copies the arrays out (into a clone of the input image)."""
        out = self.image.clone()
        fi = FakeImage.from_buffer_copy(self.fi)
        keep, ups = [], []
        for i, c in enumerate(out.comps):
            c.coef = np.ascontiguousarray(c.coef, dtype=np.int16)
            fi.coef[i] = c.coef.ctypes.data
        for j in range(len(self.ups)):
            a = np.zeros_like(self.ups[j]); ups.append(a); fi.coef_up[j] = a.ctypes.data
        self.lib.fakejpeg_store(self.h, C.byref(fi))
        for i, c in enumerate(out.comps):
            if fi.upsampled and i in (1, 2):
                c.coef = ups[i - 1]
            c.h_samp, c.v_samp = fi.h_samp[i], fi.v_samp[i]
            if c.quant is not None:
                c.quant = np.array(list(fi.quant[c.quant_tbl_no]), dtype=np.uint16)
        return out

    def close(self):
        if self.h:
            self.lib.fakejpeg_close(self.h)
            self.h = None


def run_reference(image, flags, niter, variant="scalar", threads=0, **kw):
    lib = reflib(variant)
    return run_libjpeg_boundary(lib.qsref_do_quantsmooth, image, flags | 64, niter, threads=threads, **kw)


# ---- flat restatement -------------------------------------------------------------------
class QsoComp(C.Structure):
    _fields_ = [("coef", C.c_void_p), ("wblk", C.c_uint32), ("hblk", C.c_uint32),
                ("h_samp", C.c_int), ("v_samp", C.c_int), ("has_qtbl", C.c_int),
                ("quant", C.c_uint16 * 64), ("coef_up", C.c_void_p)]


class QsoImage(C.Structure):
    _fields_ = [("ncomp", C.c_int), ("is_ycbcr", C.c_int), ("image_width", C.c_uint32),
                ("image_height", C.c_uint32), ("comp", QsoComp * 4), ("upsampled", C.c_int)]


def run_oracle(image, flags, niter, progprec=0, progress=None, threads=0):
    """The C restatement on flat arrays.  Returns (ret, result_image)."""
    from jpegqs_b200.image import JCS_YCbCr
    lib = oraclelib()
    lib.qso_set_threads(threads)
    out = image.clone()
    qi = QsoImage()
    qi.ncomp = len(out.comps)
    qi.is_ycbcr = int(out.colorspace == JCS_YCbCr)
    qi.image_width, qi.image_height = out.width, out.height
    ups = []
    for i, c in enumerate(out.comps):
        c.coef = np.ascontiguousarray(c.coef, dtype=np.int16)
        qc = qi.comp[i]
        qc.coef = c.coef.ctypes.data
        qc.wblk, qc.hblk, qc.h_samp, qc.v_samp = c.wblk, c.hblk, c.h_samp, c.v_samp
        qc.has_qtbl = int(c.quant is not None)
        if c.quant is not None:
            for k in range(64):
                qc.quant[k] = int(c.quant[k])
        if i in (1, 2) and qi.ncomp >= 3:
            a = np.zeros((out.comps[0].hblk, out.comps[0].wblk, 64), dtype=np.int16)
            ups.append(a)
            qc.coef_up = a.ctypes.data
    cb = PROGRESS_FN(progress) if progress is not None else None
    lib.qso_run.restype = C.c_int
    lib.qso_run.argtypes = [C.POINTER(QsoImage), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    ret = lib.qso_run(C.byref(qi), flags & 0x3f, niter, progprec,
                      C.cast(cb, C.c_void_p) if cb else None, None)
    for i, c in enumerate(out.comps):
        if qi.upsampled and i in (1, 2):
            c.coef = ups[i - 1]
        if qi.upsampled:
            c.h_samp = c.v_samp = 1
        if c.quant is not None:
            c.quant = np.array(list(qi.comp[i].quant), dtype=np.uint16)
    return ret, out


def images_equal(a, b):
    if len(a.comps) != len(b.comps):
        return False
    for ca, cb in zip(a.comps, b.comps):
        if ca.coef.shape != cb.coef.shape or not np.array_equal(ca.coef, cb.coef):
            return False
        if (ca.h_samp, ca.v_samp) != (cb.h_samp, cb.v_samp):
            return False
        if (ca.quant is None) != (cb.quant is None):
            return False
        if ca.quant is not None and not np.array_equal(ca.quant, cb.quant):
            return False
    return True


def diff_count(a, b):
    n = 0
    for ca, cb in zip(a.comps, b.comps):
        if ca.coef.shape != cb.coef.shape:
            return -1
        n += int(np.count_nonzero(ca.coef != cb.coef))
    return n
