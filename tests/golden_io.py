"""Load/save golden cases, look up the reference's stored outputs, and build the adversarial
inputs used by the edge-case tests."""
import hashlib
import json
import os

import numpy as np

from jpegqs_b200.image import CoefImage, Component, JCS_GRAYSCALE, JCS_YCbCr


def save_case(path, im, out, flags, niter, ret):
    d = {"width": im.width, "height": im.height, "colorspace": im.colorspace, "flags": flags,
         "niter": niter, "ret": ret, "ncomp": len(im.comps)}
    for i, (a, b) in enumerate(zip(im.comps, out.comps)):
        d[f"in{i}"] = a.coef
        d[f"out{i}"] = b.coef
        d[f"quant{i}"] = a.quant
        d[f"quant_out{i}"] = b.quant
        d[f"samp{i}"] = np.array([a.h_samp, a.v_samp, a.quant_tbl_no, b.h_samp, b.v_samp])
    np.savez_compressed(path, **d)


def load_case(path):
    z = np.load(path)
    n = int(z["ncomp"])
    comps_in, comps_out = [], []
    for i in range(n):
        s = z[f"samp{i}"]
        comps_in.append(Component(z[f"in{i}"].copy(), z[f"quant{i}"].copy(), int(s[0]), int(s[1]), int(s[2])))
        comps_out.append(Component(z[f"out{i}"].copy(), z[f"quant_out{i}"].copy(), int(s[3]), int(s[4]), int(s[2])))
    im = CoefImage(int(z["width"]), int(z["height"]), int(z["colorspace"]), comps_in)
    out = CoefImage(int(z["width"]), int(z["height"]), int(z["colorspace"]), comps_out)
    return im, out, int(z["flags"]), int(z["niter"]), int(z["ret"])


REFERENCE_OUTPUTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.json")
_reference_outputs = None


def reference_output(key):
    """What the unmodified reference gave for one test case: written by
    tests/golden/make_reference_outputs.py, outputs as SHA-256 digests (see the digest helpers)."""
    global _reference_outputs
    if _reference_outputs is None:
        with open(REFERENCE_OUTPUTS) as f:
            _reference_outputs = json.load(f)
    return _reference_outputs[key]


def digest(*chunks):
    h = hashlib.sha256()
    for c in chunks:
        h.update(c if isinstance(c, bytes) else np.ascontiguousarray(c).tobytes())
    return h.hexdigest()


def file_digest(path):
    with open(path, "rb") as f:
        return digest(f.read())


def image_digest(ret, image):
    """Everything oracle_lib.images_equal compares, plus the return code."""
    parts = [np.array([ret, len(image.comps)], dtype=np.int64)]
    for c in image.comps:
        parts += [np.array(c.coef.shape + (c.h_samp, c.v_samp, c.quant is not None), dtype=np.int64),
                  np.ascontiguousarray(c.coef, dtype=np.int16)]
        if c.quant is not None:
            parts.append(np.asarray(c.quant, dtype=np.uint16))
    return digest(*parts)


def _checker_coefs(lo, hi, q):
    """Quantized coefficients of an 8x8 1-px checkerboard lo/hi (every |d| >= 2q when q is
    small: the a3 == 0 -> NaN -> INT_MIN path of SURVEY.md 7.3 item 2)."""
    from jpegqs_b200 import synth
    px = np.where((np.add.outer(np.arange(8), np.arange(8)) & 1) == 0, lo, hi).astype(np.int64)
    return synth.quantize_blocks(px, np.full(64, q, dtype=np.uint16))[0, 0]


def adversarial_image(kind):
    rng = np.random.RandomState(99)
    W, H = 6, 5
    q = np.full(64, 2, dtype=np.uint16)
    coef = np.zeros((H, W, 64), dtype=np.int16)
    if kind == "nan":
        coef[:] = _checker_coefs(28, 228, 2)
        comps = [Component(coef, q, 1, 1, 0)]
        return CoefImage(W * 8, H * 8, JCS_GRAYSCALE, comps)
    if kind == "flat":
        coef[..., 0] = rng.randint(-60, 60, size=(H, W))
        q = np.full(64, 16, dtype=np.uint16)
        return CoefImage(W * 8, H * 8, JCS_GRAYSCALE, [Component(coef, q, 1, 1, 0)])
    if kind == "q1":                       # all quant values <= 1: iterations are skipped
        coef = rng.randint(-30, 30, size=(H, W, 64)).astype(np.int16)
        return CoefImage(W * 8, H * 8, JCS_GRAYSCALE, [Component(coef, np.ones(64, dtype=np.uint16), 1, 1, 0)])
    # three-component cases: the fault sits in component 1, so component 0 must finish
    # normally, component 1 be clamped / only de-quantized and component 2 only de-quantized
    from jpegqs_b200 import synth
    im = synth.make_image(W * 16, H * 16, "420", quality=50, seed=11)
    if kind == "badcoef":
        im.comps[1].coef[2, 1, 5] = 3000       # * q leaves [-2048, 2047] -> stop (2602-2610)
    elif kind == "bigquant":
        im.comps[1].quant = im.comps[1].quant.copy()
        im.comps[1].quant[63] = 0x800          # -> stop before the component starts (2504)
        im.comps[2].quant = im.comps[1].quant
    elif kind == "zeroquant":
        im.comps[0].quant = im.comps[0].quant.copy()
        im.comps[0].quant[10] = 0              # damaged table: 0 -> 1 for the maths, 0 for dequant
        im.comps[0].quant[63] = 0
    return im
