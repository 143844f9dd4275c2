"""The C slab engine (qs_cuda.cu run_slab / links / jpegqs_cuda_run_host_multi), the only
sharded path: one image cut into MCU-row slabs, halo rows and out-of-range masks exchanged by
CUDA kernels through peer mailboxes, the reference's `stop` logic evaluated on the device.
Everything is compared with the ORACLE (never with the product's own single-GPU run).

A box with one GPU still runs the whole exchange: several ranks may share a device (contexts
of one process connected "locally", or two processes connected through CUDA IPC handles)."""
import multiprocessing as mp
import os

import numpy as np
import pytest

import jpegqs_b200 as qs
import oracle_lib as ol
from golden_io import adversarial_image
from jpegqs_b200 import multigpu as mg
from jpegqs_b200.image import CoefImage, Component

pytestmark = pytest.mark.gpu


def cut(im, world):
    """[(slab image, row0 per component)] for `world` ranks - the geometry of
    jpegqs_cuda_run_host_multi (contiguous MCU rows, sizes differing by at most one)."""
    maxv = max(c.v_samp for c in im.comps)
    mcu_total = -(-im.height // (8 * maxv))
    out = []
    for m in mg.split_mcu_rows(mcu_total, world):
        comps, row0 = [], []
        for c in im.comps:
            r0, r1 = mg.comp_block_rows(m, c.v_samp, c.hblk)
            comps.append(Component(c.coef[r0:r1].copy(), None if c.quant is None else c.quant.copy(),
                                   c.h_samp, c.v_samp, c.quant_tbl_no))
            row0.append(r0)
        out.append((CoefImage(im.width, im.height, im.colorspace, comps), row0))
    return out


def glue(im, parts, ups, upsampled):
    """Whole-image result from the ranks' slabs."""
    out = im.clone()
    for k, c in enumerate(out.comps):
        if upsampled and k in (1, 2):
            c.coef = np.concatenate([u[k - 1] for u in ups], axis=0)
        else:
            c.coef = np.concatenate([p.comps[k].coef for p, _ in parts], axis=0)
        if upsampled:
            c.h_samp = c.v_samp = 1
        c.quant = parts[0][0].comps[k].quant
    return out


@pytest.fixture(scope="module")
def ctx():
    c = qs.cuda.QsContext(0)
    yield c
    c.close()


CASES = [(200, 136, "420", 0, 3), (200, 136, "420", 1, 2), (256, 200, "420", 3, 2), (256, 200, "420", 7, 3),
         (250, 130, "444", 7, 2), (160, 400, "gray", 1, 3), (136, 120, "422", 3, 2), (136, 120, "440", 0, 3),
         (200, 136, "420", 8, 2), (200, 136, "420", 8 | 7, 1), (90, 50, "420", 7, 2), (200, 136, "420", 16, 2),
         (128, 64, "422", 7, 2), (48, 40, "gray", 16, 3)]


@pytest.mark.parametrize("w,h,ss,flags,niter", CASES)
def test_one_rank_run_slab_matches_oracle(ctx, w, h, ss, flags, niter):
    """world = 1: the slab engine is a complete do_quantsmooth with the stop logic on the device."""
    im = qs.synth.make_image(w, h, ss)
    (slab, row0), = cut(im, 1)
    ret, ups_flag, ups = ctx.run_slab(None, slab, 0, 1, row0, [c.hblk for c in im.comps], flags, niter)
    oret, want = ol.run_oracle(im, flags, niter)
    assert ret == oret
    assert ol.images_equal(glue(im, [(slab, row0)], [ups], ups_flag), want)


@pytest.mark.parametrize("kind", ["badcoef", "bigquant", "zeroquant", "nan", "q1"])
@pytest.mark.parametrize("flags", [0, 7])
def test_one_rank_stop_logic_on_the_device(ctx, kind, flags):
    im = adversarial_image(kind)
    (slab, row0), = cut(im, 1)
    ret, ups_flag, ups = ctx.run_slab(None, slab, 0, 1, row0, [c.hblk for c in im.comps], flags, 2)
    oret, want = ol.run_oracle(im, flags, 2)
    assert ret == oret
    assert ol.images_equal(glue(im, [(slab, row0)], [ups], ups_flag), want)


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [k % have for k in range(n)]       # ranks share devices when the box has fewer


def _multi(world):
    os.environ["JPEGQS_MIN_BLOCKS_PER_GPU"] = "1"                 # shard even tiny images
    try:
        return qs.cuda.QsMulti(_devices(world))
    finally:
        del os.environ["JPEGQS_MIN_BLOCKS_PER_GPU"]


def _multi_matches_oracle(m, im, flags, niter):
    ret, out = m.do_quantsmooth(im, flags, niter)
    oret, want = ol.run_oracle(im, flags, niter)
    assert ret == oret
    assert ol.images_equal(out, want), f"{ol.diff_count(out, want)} coefficients differ"


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("w,h,ss,flags,niter", CASES)
def test_run_host_multi_matches_oracle(world, w, h, ss, flags, niter):
    m = _multi(world)
    try:
        im = qs.synth.make_image(w, h, ss)
        assert m.plan(im) == world
        _multi_matches_oracle(m, im, flags, niter)
    finally:
        m.close()


@pytest.mark.parametrize("world,flags", [(2, 0), (3, 1), (5, 0), (3, 8)])
def test_slabs_are_shard_invariant(world, flags):
    """13 MCU rows over up to 5 ranks: slabs of 2 and 3 MCU rows, up to four interior boundaries."""
    m = _multi(world)
    try:
        im = qs.synth.make_image(256, 208, "420")
        assert m.plan(im) == world
        _multi_matches_oracle(m, im, flags, 2)
    finally:
        m.close()


@pytest.mark.parametrize("flags,niter", [(0, 3), (7, 2), (1, 1)])
def test_multi_stop_reaches_every_rank(flags, niter):
    """An out-of-range coefficient in the LAST rank's slab: the first rank must leave that
    component alone as well (quantsmooth.h:2602-2610), which it only learns from the exchange."""
    m = _multi(3)
    try:
        for comp, pos in ((0, -1), (1, -1), (2, 0), (1, 0)):
            im = qs.synth.make_image(160, 240, "420")
            c = im.comps[comp]
            c.coef[pos, 2, 1] = 3000
            ret, out = m.do_quantsmooth(im, flags, niter)
            oret, want = ol.run_oracle(im, flags, niter)
            assert ret == oret and oret != 0
            assert ol.images_equal(out, want), (comp, pos)
        for kind in ("bigquant", "zeroquant"):
            im = adversarial_image(kind)
            ret, out = m.do_quantsmooth(im, flags, niter)
            oret, want = ol.run_oracle(im, flags, niter)
            assert ret == oret and ol.images_equal(out, want), kind
    finally:
        m.close()


def test_multi_keeps_small_images_on_one_device():
    m = qs.cuda.QsMulti(_devices(2))
    try:
        im = qs.synth.make_image(640, 480, "420")
        assert m.plan(im) == 1                       # one wave of the smoothing kernel is 75 776 blocks
        ret, out = m.do_quantsmooth(im, 0, 2)
        assert ol.images_equal(out, ol.run_oracle(im, 0, 2)[1])
    finally:
        m.close()


# ---- ranks in different processes: CUDA IPC mailboxes -------------------------------------------
def _ipc_rank(rank, world, w, h, ss, flags, niter, reps, conns, result):
    import torch
    dev = rank % torch.cuda.device_count()
    ctx = qs.cuda.QsContext(dev)
    im = qs.synth.make_image(w, h, ss)
    slab, row0 = cut(im, world)[rank]
    link = qs.cuda.QsLink(ctx, rank, world, max(c.wblk for c in im.comps))
    mine = link.export()
    for c in conns[rank]["out"]:
        c.send(mine)
    handles = [None] * world
    handles[rank] = mine
    for src, c in conns[rank]["in"]:
        handles[src] = c.recv()
    link.connect_ipc(handles)
    outs = []
    for rep in range(reps):
        s = slab.clone()
        ret, ups_flag, ups = ctx.run_slab(link, s, rank, world, row0, [c.hblk for c in im.comps], flags, niter)
        outs.append((ret, ups_flag, [c.coef for c in s.comps], ups))
    result.put((rank, outs))
    link.close()
    ctx.close()


def run_ranks_in_processes(world, w, h, ss, flags, niter, reps):
    """One process per rank (sharing devices on a box with fewer GPUs), mailboxes connected through
    CUDA IPC handles.  Returns {rank: [(ret, upsampled, coefs, up arrays) per repetition]}."""
    sp = mp.get_context("spawn")
    pipes = {(a, b): sp.Pipe(duplex=False) for a in range(world) for b in range(world) if a != b}
    conns = [{"out": [pipes[(r, d)][1] for d in range(world) if d != r],
              "in": [(s, pipes[(s, r)][0]) for s in range(world) if s != r]} for r in range(world)]
    result = sp.Queue()
    procs = [sp.Process(target=_ipc_rank, args=(r, world, w, h, ss, flags, niter, reps, conns, result))
             for r in range(world)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(world):
        rank, outs = result.get(timeout=300)
        got[rank] = outs
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    return got


@pytest.mark.parametrize("w,h,ss,flags,niter", [(320, 272, "420", 0, 3), (320, 272, "420", 7, 2), (256, 200, "444", 1, 2)])
def test_two_processes_over_cuda_ipc(w, h, ss, flags, niter):
    world = 2
    got = run_ranks_in_processes(world, w, h, ss, flags, niter, 2)   # twice: sequence numbers carry over
    im = qs.synth.make_image(w, h, ss)
    oret, want = ol.run_oracle(im, flags, niter)
    for rep in range(2):
        assert all(got[r][rep][0] == oret for r in range(world))
        upsampled = got[0][rep][1]
        out = im.clone()
        for k, c in enumerate(out.comps):
            if upsampled and k in (1, 2):
                c.coef = np.concatenate([got[r][rep][3][k - 1] for r in range(world)], axis=0)
            else:
                c.coef = np.concatenate([got[r][rep][2][k] for r in range(world)], axis=0)
        for a, b in zip(out.comps, want.comps):
            assert a.coef.shape == b.coef.shape and np.array_equal(a.coef, b.coef), (rep, flags)


# ---- full BASELINE sizes against the oracle (whole image, every byte) ---------------------------
@pytest.mark.parametrize("w,h,flags,niter", [(3840, 2160, 0, 3), (7680, 4320, 0, 3), (7680, 4320, 7, 3)])
def test_whole_image_parity_at_baseline_sizes(ctx, w, h, flags, niter):
    """BASELINE configs 2 and 3 (+ the headline shape): EVERY output coefficient against the
    oracle (OpenMP, all host threads), through the host entry point with block-row tables."""
    im = qs.synth.make_image(w, h, "420")
    ret, out = ctx.do_quantsmooth(im, flags, niter)
    oret, want = ol.run_oracle(im, flags, niter, threads=0)
    assert ret == oret == 0
    assert ol.images_equal(out, want), f"{ol.diff_count(out, want)} coefficients differ"


def test_sharded_large_image_parity_vs_oracle():
    """>= 4096^2, q4 n5 and q6 (BASELINE config 5's recipe at a size the oracle finishes in
    seconds), sharded over 2 ranks with the kernel exchange, against the oracle."""
    m = qs.cuda.QsMulti(_devices(2))
    try:
        im = qs.synth.make_image(4096, 4096, "420")
        assert m.plan(im) == 2
        for flags, niter in ((1, 5), (7, 3)):
            ret, out = m.do_quantsmooth(im, flags, niter)
            oret, want = ol.run_oracle(im, flags, niter, threads=0)
            assert ret == oret == 0
            assert ol.images_equal(out, want), (flags, ol.diff_count(out, want))
    finally:
        m.close()


def test_batch_of_1080p_images_against_the_oracle(ctx):
    """BASELINE config 4's shape (1920x1080 4:2:0, q3 n3) through run_batch: 16 images checked."""
    ims = [qs.synth.make_image(1920, 1080, "420", seed=100 + k) for k in range(16)]
    rets, outs = ctx.run_batch_host(ims, 0, 3)
    for im, ret, out in zip(ims, rets, outs):
        oret, want = ol.run_oracle(im, 0, 3, threads=0)
        assert ret == oret and ol.images_equal(out, want)
