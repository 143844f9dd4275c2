"""GPU edge cases, the libjpeg-facing C entry point, the batch entry point, and
size-independent properties at BASELINE.json's full sizes."""
import ctypes as C
import hashlib

import numpy as np
import pytest

import jpegqs_b200 as qs
import oracle_lib as ol
from golden_io import adversarial_image, image_digest, reference_output

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = qs.cuda.QsContext(0)
    yield c
    c.close()


def _same(ctx, im, flags, niter, **kw):
    ret, out = ctx.do_quantsmooth(im, flags, niter, **kw)
    oret, oout = ol.run_oracle(im, flags, niter)
    assert ret == oret
    assert ol.images_equal(out, oout), f"{ol.diff_count(out, oout)} coefficients differ"
    return out


@pytest.mark.parametrize("kind,flags,niter", [("nan", 0, 1), ("nan", 1, 2), ("badcoef", 0, 2), ("bigquant", 0, 2),
                                              ("zeroquant", 0, 2), ("flat", 1, 2), ("q1", 0, 3),
                                              ("badcoef", 7, 2), ("bigquant", 7, 1), ("zeroquant", 7, 2)])
def test_adversarial(ctx, kind, flags, niter):
    _same(ctx, adversarial_image(kind), flags, niter)


def test_niter_zero_and_clamping_of_niter(ctx):
    im = qs.synth.make_image(64, 48, "420")
    ret, out = ctx.do_quantsmooth(im, 0, 0)          # early return: nothing touched (2458)
    assert ret == 0 and ol.images_equal(out, im)
    _same(ctx, im, 4, 0)                             # UPSAMPLE_UV alone still runs (2458, 2495)
    _same(ctx, im, 0, -5)
    ret, out = ctx.do_quantsmooth(im, 0, 1000)       # clamped to JPEGQS_ITER_MAX
    ret2, out2 = ctx.do_quantsmooth(im, 0, 100)
    assert ol.images_equal(out, out2)


@pytest.mark.parametrize("w,h,ss,flags,niter,quality", [
    (256, 128, "420", 8 | 1, 3, 30),       # -q 0
    (250, 130, "420", 8 | 3, 2, 20),       # -q 1 (JOINT_YUV predictor, then rebalance only)
    (256, 128, "420", 8 | 7, 2, 40),       # -q 2 (+ UPSAMPLE_UV)
    (128, 64, "gray", 8, 3, 10),
    (256, 128, "444", 8 | 7, 2, 50),
    (64, 48, "420", 8 | 16, 2, 30),
    (1920, 1080, "420", 8 | 1, 3, 25),
])
def test_low_quality(ctx, w, h, ss, flags, niter, quality):
    """LOW_QUALITY (q0-2): the scalar branch's int truncation is the contract (SURVEY.md 4)."""
    _same(ctx, qs.synth.make_image(w, h, ss, quality=quality), flags, niter)


def test_component_without_table_and_four_components(ctx):
    im = qs.synth.make_image(64, 48, "420")
    im.comps[1].quant = None
    _same(ctx, im, 1, 2)
    im = qs.synth.make_image(64, 48, "444")
    im.colorspace = qs.JCS_RGB                        # not YCbCr: all components are "luma"
    _same(ctx, im, 7 | 32, 2)


def test_progress_sequence_and_cancel(ctx):
    im = qs.synth.make_image(96, 80, "420")
    seq_o, seq_g = [], []
    ol.run_oracle(im, 3, 3, progprec=7, progress=lambda d, cur, mx: seq_o.append((cur, mx)) or 0)
    ret, out = ctx.do_quantsmooth(im, 3, 3, progprec=7, progress=lambda cur, mx: seq_g.append((cur, mx)) or 0)
    assert seq_g == seq_o and len(seq_g) > 2
    _, want = ol.run_oracle(im, 3, 3)
    assert ol.images_equal(out, want)
    s1, s2 = [], []
    r1, o1 = ol.run_oracle(im, 0, 3, progprec=7, progress=lambda d, cur, mx: (s1.append(cur), 5 if len(s1) >= 2 else 0)[1])
    r2, o2 = ctx.do_quantsmooth(im, 0, 3, progprec=7, progress=lambda cur, mx: (s2.append(cur), 5 if len(s2) >= 2 else 0)[1])
    assert r1 == r2 == 5 and s1 == s2
    assert ol.images_equal(o1, o2)


BOUNDARY_CASES = [(0, 3, "420"), (7, 2, "420"), (3, 2, "444"), (1, 1, "gray")]


@pytest.mark.parametrize("flags,niter,ss", BOUNDARY_CASES)
def test_libjpeg_facing_entry_point(flags, niter, ss):
    """do_quantsmooth(j_decompress_ptr, jvirt_barray_ptr*, jpegqs_control_t*) through the
    fake libjpeg front end, rows scattered in memory like libjpeg's virtual arrays; the
    reference's result through the same front end is stored (reference_outputs())."""
    lib = qs.cuda.load()
    im = qs.synth.make_image(120, 72, ss)
    ret, out = ol.run_libjpeg_boundary(lib.do_quantsmooth, im, flags | 64, niter, scatter_rows=True)
    oret, oout = ol.run_oracle(im, flags, niter)
    assert ret == oret and ol.images_equal(out, oout)
    assert image_digest(ret, out) == reference_output(f"libjpeg_boundary/{flags},{niter},{ss}")


def reference_outputs(tmpdir):
    return {f"libjpeg_boundary/{flags},{niter},{ss}":
            image_digest(*ol.run_reference(qs.synth.make_image(120, 72, ss), flags, niter, scatter_rows=True))
            for flags, niter, ss in BOUNDARY_CASES}


def test_batch_entry_point(ctx):
    ims = [qs.synth.make_image(1920 // 4, 1080 // 4, "420", seed=s) for s in range(5)]
    ims.append(adversarial_image("badcoef"))
    ims.append(qs.synth.make_image(64, 64, "gray", quality=80))
    for flags in (0, 7):
        rets, outs = ctx.run_batch_host(ims, flags, 2)
        for im, r, o in zip(ims, rets, outs):
            wr, want = ol.run_oracle(im, flags, 2)
            assert r == wr and ol.images_equal(o, want)


def test_batch_larger_than_one_launch(ctx):
    """More components than one launch carries (QS_MAX_JOBS = 1024): split into sub-batches."""
    base = [qs.synth.make_image(48, 32, "420", seed=s) for s in range(4)]
    ims = [base[i % 4] for i in range(400)]
    rets, outs = ctx.run_batch_host(ims, 0, 1)
    wants = [ol.run_oracle(b, 0, 1)[1] for b in base]
    assert not any(rets)
    for i, o in enumerate(outs):
        assert ol.images_equal(o, wants[i % 4])


DEFAULT_MERGE = 1        # csrc/qs_cuda.cu tune_merge


def test_tuning_variants_are_bit_identical(ctx):
    """The shipped library carries one lock-step configuration (the others live behind
    -DQS_EXPERIMENTS); what can still vary is the chunk schedule: 1..4 coefficients per chunk,
    with and without uniform-quant chunks.  Every schedule gives the oracle's bytes."""
    im = qs.synth.make_image(320, 240, "420")
    want = {f: ol.run_oracle(im, f, 2)[1] for f in (0, 1)}
    try:
        for merge in (0, 1):                          # key 8: edge coefficients in "mixed" chunks
            ctx.set_tuning(8, merge)
            for uni in (0, 1):
                for maxn in (1, 2, 3, 4):
                    ctx.set_tuning(1, maxn); ctx.set_tuning(5, uni)
                    for f in (0, 1):
                        _, out = ctx.do_quantsmooth(im, f, 2)
                        assert ol.images_equal(out, want[f]), (merge, uni, maxn, f)
        ctx.set_tuning(8, 1); ctx.set_tuning(1, 4); ctx.set_tuning(5, 1)
        for w, h, ss, f in ((250, 130, "444", 7), (160, 400, "gray", 1), (136, 120, "422", 3), (200, 136, "420", 0)):
            im2 = qs.synth.make_image(w, h, ss)
            ret, out = ctx.do_quantsmooth(im2, f, 2)
            oret, o = ol.run_oracle(im2, f, 2)
            assert ret == oret and ol.images_equal(out, o), (w, h, ss, f)
        with pytest.raises(qs.cuda.QsError):
            ctx.set_tuning(0, 0)                      # free-running warps: experiments build only
    finally:
        ctx.set_tuning(1, 4); ctx.set_tuning(5, 1); ctx.set_tuning(8, DEFAULT_MERGE)


# ---- full BASELINE sizes: size-independent properties (the oracle would take minutes) ----
def _interval_property(im, out):
    """Every output coefficient stays inside the quantization interval of its input:
    |out - in*q| <= q/2 (quantsmooth.h:1551-1564), clamped to +-1023 (2670-2689)."""
    for a, b in zip(im.comps, out.comps):
        q = a.quant.astype(np.int32)
        a0 = a.coef.astype(np.int32) * q
        lo = np.clip(a0 - (q >> 1), -1023, 1023)
        hi = np.clip(a0 + (q >> 1), -1023, 1023)
        assert np.all((b.coef >= lo) & (b.coef <= hi))
        assert np.array_equal(b.quant, np.ones(64, dtype=np.uint16))


def test_8k_q3_properties_and_row_band_parity(ctx):
    im = qs.synth.make_image(7680, 4320, "420")                     # BASELINE headline shape
    ret, out = ctx.do_quantsmooth(im, 0, 3)
    assert ret == 0
    _interval_property(im, out)
    # a horizontal band of the image smoothed on its own differs from the full run only next
    # to the cut (Jacobi dependence reaches 1 block row per iteration): compare the interior
    band = qs.synth.make_image(7680, 4320, "420", mcu_rows=(100, 112))
    band.height = 12 * 16
    _, bo = ol.run_oracle(band, 0, 3, threads=0)
    for k, (c, b) in enumerate(zip(out.comps, bo.comps)):
        r0 = 100 * (2 if k == 0 else 1)
        m = 3                                                        # niter block rows of margin
        assert np.array_equal(c.coef[r0 + m:r0 + b.hblk - m], b.coef[m:b.hblk - m]), k


def test_8k_q3_shard_invariance_over_processes(ctx):
    """The headline shape over 4 ranks of the C slab engine, one process per rank (sharing
    devices on a box with fewer GPUs, connected through CUDA IPC), against the single-device run."""
    from test_gpu_slab_engine import run_ranks_in_processes
    im = qs.synth.make_image(7680, 4320, "420")
    _, want = ctx.do_quantsmooth(im, 0, 3)
    got = run_ranks_in_processes(4, 7680, 4320, "420", 0, 3, 1)
    assert all(got[r][0][0] == 0 for r in range(4))
    for k, c in enumerate(want.comps):
        assert np.array_equal(np.concatenate([got[r][0][2][k] for r in range(4)], axis=0), c.coef), k


def test_8k_q6_properties(ctx):
    im = qs.synth.make_image(7680, 4320, "420")                     # BASELINE config 3
    ret, out = ctx.do_quantsmooth(im, 7, 3)
    assert ret == 0
    assert [c.coef.shape for c in out.comps] == [(540, 960, 64)] * 3
    assert all(c.h_samp == 1 and c.v_samp == 1 for c in out.comps)
    _interval_property(qs.CoefImage(im.width, im.height, im.colorspace, im.comps[:1]),
                       qs.CoefImage(im.width, im.height, im.colorspace, out.comps[:1]))
    # band parity: luma differs within 3 block rows of the cut; chroma is predicted from the
    # luma plane and then re-sampled to luma resolution, so its disturbed zone is wider
    band = qs.synth.make_image(7680, 4320, "420", mcu_rows=(40, 64))
    band.height = 24 * 16
    _, bo = ol.run_oracle(band, 7, 3, threads=0)
    for k, (c, b) in enumerate(zip(out.comps, bo.comps)):
        m = 3 if k == 0 else 16
        assert np.array_equal(c.coef[80 + m:128 - m], b.coef[m:48 - m]), k
