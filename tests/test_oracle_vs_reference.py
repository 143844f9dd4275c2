"""Pins the C restatement (oracle/qs_oracle.c) against the UNMODIFIED reference
(oracle/_ref/libqsref_scalar.so, the -DNO_SIMD build of the reference's quantsmooth.h).
What the reference gives for every case below is stored in tests/golden/reference_outputs.json
(reference_outputs() computes it; tests/golden/make_reference_outputs.py writes it), so the
tests need no reference build."""
import numpy as np
import pytest

import jpegqs_b200 as qs
import oracle_lib as ol
from golden_io import adversarial_image, digest, image_digest, reference_output


def test_natural_order_and_refresh_points():
    # reference idct.h:24-33 / quantsmooth.h:313-322: the refresh flag is set exactly at
    # the first-visited coefficient of each anti-diagonal in reverse zig-zag order
    zz = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20,
          13, 6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52,
          45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63]
    assert sorted(zz) == list(range(64))
    refresh = {2, 4, 6, 8, 15, 24, 31, 40, 47, 56, 58, 60, 62, 63}      # the table's 1s, minus DC
    got = set()
    for k in range(63, 0, -1):
        i = zz[k]
        if k == 63 or (zz[k + 1] // 8 + zz[k + 1] % 8) != (i // 8 + i % 8):
            got.add(i)
    assert got == refresh


def _idct_islow(idct):
    """Digests of the pixels idct makes of 200 random blocks, one per coefficient scale."""
    rng = np.random.RandomState(1)
    out = []
    for scale in (8, 200, 2047):
        pixels = []
        for _ in range(200):
            c = rng.randint(-scale, scale + 1, size=64).astype(np.int16)
            if rng.rand() < 0.3:
                c[rng.rand(64) < 0.8] = 0
            a = np.zeros((8, 24), dtype=np.uint8)
            idct(c.ctypes.data, a.ctypes.data, 24)
            pixels.append(a)
        out.append(digest(*pixels))
    return out


def test_idct_islow_exact():
    assert _idct_islow(ol.oraclelib().qso_idct_islow) == reference_output("idct_islow")


def _float_dct(fn):
    rng = np.random.RandomState(2)
    out = []
    for _ in range(300):
        x = (rng.rand(64).astype(np.float32) - 0.5) * np.float32(rng.choice([1, 255, 4096]))
        a = np.zeros(64, dtype=np.float32)
        fn(x.copy().ctypes.data, a.ctypes.data)
        out.append(a.view(np.uint32))
    return digest(*out)


def test_float_dcts_bit_exact():
    orc = ol.oraclelib()
    assert _float_dct(orc.qso_fdct_float) == reference_output("fdct_float")
    assert _float_dct(orc.qso_idct_float) == reference_output("idct_float")


def _tables(fn, flags):
    a = np.zeros((64, 272 if flags else 160), dtype=np.float32)
    fn(flags, a.ctypes.data)
    return digest(a.view(np.uint32))


@pytest.mark.parametrize("flags", [0, 1])
def test_tables_bit_exact(flags):
    assert ol.oraclelib().qso_table_size(flags) == (272 if flags else 160)
    assert _tables(ol.oraclelib().qso_tables, flags) == reference_output(f"tables/{flags}")


def test_orig_coef_exhaustive_vs_reference_formula():
    # plain form (quantsmooth.h:338-341) over the whole valid range, vectorised
    orc = ol.oraclelib()
    c = np.arange(-0x4000, 0x4000, dtype=np.int64)
    for q in list(range(1, 300)) + [511, 512, 513, 1023, 1024, 2047]:
        h = q >> 1
        n = c + np.where(c < 0, -h, h)
        want = np.sign(n) * (np.abs(n) // q) * q
        for cc in (-0x4000, -q, -h - 1, -h, -1, 0, 1, h, h + 1, q, 0x3fff):
            assert orc.qso_orig_coef(int(cc), q) == int(want[cc + 0x4000])


CASES = [
    (512, 512, "gray", 0, 3, 50),            # BASELINE config 1 (CPU scalar plumbing)
    (256, 128, "420", 0, 3, 50), (250, 130, "420", 0, 2, 92), (256, 128, "420", 1, 2, 50),
    (256, 128, "420", 3, 2, 50), (256, 128, "420", 7, 2, 50), (200, 120, "420", 7, 3, 75),
    (256, 128, "444", 7, 2, 50), (256, 128, "422", 7, 2, 50), (248, 136, "440", 7, 2, 75),
    (128, 64, "420", 16, 2, 50), (128, 64, "420", 33, 2, 50), (128, 64, "420", 6, 0, 50),
    (128, 64, "420", 0, 0, 50), (8, 8, "gray", 0, 3, 50), (128, 64, "420", 5, 1, 30),
    (256, 128, "420", 9, 3, 30), (250, 130, "420", 11, 2, 20), (256, 128, "420", 15, 2, 40),
    (128, 64, "gray", 8, 3, 10), (256, 128, "444", 15, 2, 50), (64, 48, "420", 24, 2, 30),
]


@pytest.mark.parametrize("w,h,ss,flags,niter,quality", CASES)
def test_driver_matches_reference(w, h, ss, flags, niter, quality):
    im = qs.synth.make_image(w, h, ss, quality=quality)
    assert image_digest(*ol.run_oracle(im, flags, niter)) == reference_output(f"driver/{w},{h},{ss},{flags},{niter},{quality}")


ADVERSARIAL = [("nan", 0, 1), ("badcoef", 0, 2), ("bigquant", 0, 2), ("zeroquant", 0, 2), ("flat", 1, 2), ("q1", 0, 3),
               ("badcoef", 7, 2), ("bigquant", 7, 1)]


@pytest.mark.parametrize("kind,flags,niter", ADVERSARIAL)
def test_adversarial_matches_reference(kind, flags, niter):
    im = adversarial_image(kind)
    assert image_digest(*ol.run_oracle(im, flags, niter)) == reference_output(f"adversarial/{kind},{flags},{niter}")


def test_nan_case_moves_coefficients():
    # SURVEY.md 7.3 item 2: with a3 == 0 the x86 conversion yields INT_MIN and coefficients
    # move to their clamp edge; a conversion that yields 0 would leave them unchanged
    im = adversarial_image("nan")
    _, out = ol.run_oracle(im, 0, 1)
    deq = im.comps[0].coef.astype(np.int32) * im.comps[0].quant.astype(np.int32)
    assert np.count_nonzero(out.comps[0].coef != deq) > 0


def test_non_contiguous_rows_and_threads():
    """The reference's result with scattered rows and 3 threads (stored) is the restatement's
    with 1 and with 3 threads."""
    im = qs.synth.make_image(96, 80, "420")
    want = reference_output("scattered_rows_3_threads")
    for threads in (1, 3):
        assert image_digest(*ol.run_oracle(im, 7, 2, threads=threads)) == want


def _progress(run):
    """The progress sequence of a full run, then a run cancelled at the second callback."""
    im = qs.synth.make_image(96, 80, "420")
    seq = []
    run(im, 0, 3, progprec=7, progress=lambda d, cur, mx: seq.append([cur, mx]) or 0)
    cancelled = []
    ret, out = run(im, 0, 3, progprec=7,
                   progress=lambda d, cur, mx: (cancelled.append(cur), 5 if len(cancelled) >= 2 else 0)[1])
    return {"sequence": seq, "cancelled": cancelled, "cancelled_ret": ret, "cancelled_result": image_digest(ret, out)}


def test_progress_sequence_and_cancel():
    want = reference_output("progress")
    assert len(want["sequence"]) > 2 and want["cancelled_ret"] == 5
    assert _progress(ol.run_oracle) == want


def _sweep():
    """The same seeded sweep the GPU parity test runs (tests/test_gpu_parity.py)."""
    rng = np.random.RandomState(20260923)
    modes = ["gray", "444", "422", "420", "440"]
    for case in range(48):
        ss = modes[rng.randint(len(modes))]
        w, h = int(rng.randint(8, 180)), int(rng.randint(8, 140))
        quality = int(rng.choice([3, 10, 25, 50, 75, 90, 97, 100]))
        flags = int(rng.randint(0, 64))
        if (flags & 4) and ss in ("420", "422", "440"):
            w = max(16, w // 16 * 16)
        niter = int(rng.randint(1, 4))
        im = qs.synth.make_image(w, h, ss, quality=quality, seed=1000 + case, noise=int(rng.randint(0, 12)))
        yield (case, w, h, ss, quality, flags, niter), im


def test_randomized_sweep_matches_reference():
    """The sweep, here pinning the checker itself against the unmodified reference."""
    want = reference_output("sweep")
    for (case, w, h, ss, quality, flags, niter), im in _sweep():
        assert image_digest(*ol.run_oracle(im, flags, niter)) == want[case], (case, w, h, ss, quality, flags, niter)


def reference_outputs(tmpdir):
    """What the reference gives for every case above, keyed as the tests look it up."""
    ref = ol.reflib()
    out = {"idct_islow": _idct_islow(ref.qsref_idct_islow)}
    out["fdct_float"], out["idct_float"] = _float_dct(ref.qsref_fdct_float), _float_dct(ref.qsref_idct_float)
    for flags in (0, 1):
        out[f"tables/{flags}"] = _tables(ref.qsref_tables, flags)
    for w, h, ss, flags, niter, quality in CASES:
        im = qs.synth.make_image(w, h, ss, quality=quality)
        out[f"driver/{w},{h},{ss},{flags},{niter},{quality}"] = image_digest(*ol.run_reference(im, flags, niter))
    for kind, flags, niter in ADVERSARIAL:
        out[f"adversarial/{kind},{flags},{niter}"] = image_digest(*ol.run_reference(adversarial_image(kind), flags, niter))
    im = qs.synth.make_image(96, 80, "420")
    out["scattered_rows_3_threads"] = image_digest(*ol.run_reference(im, 7, 2, scatter_rows=True, threads=3))
    assert out["scattered_rows_3_threads"] == image_digest(*ol.run_reference(im, 7, 2, threads=1))
    out["progress"] = _progress(ol.run_reference)
    out["sweep"] = [image_digest(*ol.run_reference(im, c[-2], c[-1])) for c, im in _sweep()]
    return out
