#!/usr/bin/env python
"""bench.py - the hot path's benchmark.

    python bench.py --gpus 1 --steps K --warmup W            # B200 arm
    python bench.py --impl reference --steps K --warmup W    # reference CPU arm
    torchrun --nproc-per-node N ... bench.py --gpus N ...    # MCU-row sharded, weak scaling
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's result

--dump-outputs DIR writes DIR/ret.npy (the call's return code) and DIR/coef<k>.npy: a fixed, seeded
sample of a quarter of component k's smoothed 8x8 blocks (float32, shape (blocks, 64); exact for the
int16 coefficients).  The input is the same seeded image in every run, so two builds (or the two arms)
can be compared array for array.  Ranks of a sharded run prefix their files with rank<r>_.  The reference
arm's AVX-512 build is called with JPEGQS_TRANSCODE and so returns re-quantized coefficients; the B200
arm and the reference arm's C port return de-quantized ones.

A "step" is one complete do_quantsmooth pass (all components, all iterations) over one
synthetic image.  N=1 workload: BASELINE.json's metric configuration, 7680x4320 YCbCr
4:2:0, q=3 (flags 0), niter=3.  N>1: the same image stacked N times vertically
(7680 x 4320*N), sharded by MCU rows with one halo pixel row per component exchanged over
NCCL between the IDCT and smoothing passes of every iteration (weak scaling).

Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mpixels/sec at q=3 niter=3 (8K 4:2:0); achieved HBM GB/s vs peak"
WIDTH, HEIGHT, SUBSAMPLING, FLAGS, NITER, QUALITY, SEED = 7680, 4320, "420", 0, 3, 50, 12345
ALGO_BYTES_PER_BLOCK_ITER = 256          # SURVEY.md 8d: 128 B coefficient read + 128 B write
DUMP_SHARE = 4                           # --dump-outputs keeps 1 block in DUMP_SHARE: 50 MB at 8K 4:2:0


def dump_outputs(d, ret, coefs, prefix="", world=1):
    """ret and a seeded sample of whole blocks of each component's coefficients, as float32 .npy."""
    os.makedirs(d, exist_ok=True)
    rng = np.random.RandomState(SEED)
    np.save(os.path.join(d, prefix + "ret.npy"), np.array([ret], dtype=np.float64))
    for k, c in enumerate(coefs):
        blocks = np.asarray(c).reshape(-1, 64)
        keep = np.sort(rng.choice(len(blocks), len(blocks) // (DUMP_SHARE * world), replace=False))
        np.save(os.path.join(d, f"{prefix}coef{k}.npy"), blocks[keep].astype(np.float32))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.t0 = self.t1 = None        # perf_counter window of the timed region

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [ln for (t, ln) in self.lines if self.t0 is not None and self.t0 <= t <= self.t1 + 0.03]
        scope = "timed region"
        if len(inside) < 2:                 # region shorter than the sampling period: use the
            inside = [ln for (t, ln) in self.lines if self.t0 is None or t >= self.t0 - 0.5]   # loaded phase
            scope = "timed region + end-to-end phase"
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, name in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "scope": scope, "reasons": sorted(reasons)}


def make_workload(world, rank):
    import jpegqs_b200 as qs
    mcu_total = (HEIGHT * world + 15) // 16
    from jpegqs_b200.multigpu import split_mcu_rows
    rng = split_mcu_rows(mcu_total, world)[rank]
    im = qs.synth.make_image(WIDTH, HEIGHT * world, SUBSAMPLING, quality=QUALITY, seed=SEED,
                             mcu_rows=None if world == 1 else rng)
    return im, rng, mcu_total


def cpu_reference_time(im, threads=0, runs=5):
    """The reference's own AVX-512+OpenMP do_quantsmooth (oracle/_ref, built from the
    unmodified sources) - or, if that object is absent, the scalar C port with OpenMP -
    timed on this box's host cores.  Returns (seconds_median, kind, cores, how)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    ol.ensure_built()
    if ol.have_ref("avx512"):
        lib = ol.reflib("avx512")
        cores = lib.qsref_num_procs()
        best = None
        # the reference's default is all processors (opts.threads = 0); on many-core hosts
        # fewer threads can be faster, so the best of {all, 1/2, 1/4} is reported (fair to it)
        for thr in sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True):
            times = []
            for i in range(runs + 1):
                lib.qsref_take_log()
                ol.run_reference(im, FLAGS | (8 << 16), NITER, variant="avx512", threads=thr)
                log = lib.qsref_take_log().decode()
                ms = [float(l.split(":")[1].replace("ms", "")) for l in log.splitlines() if l.startswith("quantsmooth:")]
                if i and ms:
                    times.append(ms[-1] / 1e3)
            med = statistics.median(times)
            if best is None or med < best[0]:
                best = (med, thr)
        return best[0], "reference", best[1], ("reference's own timer ('quantsmooth: ..ms'), AVX-512 + OpenMP, "
                                              f"best of thread counts all/half/quarter of {cores} processors")
    lib = ol.oraclelib()
    cores = lib.qso_num_procs()
    times = []
    for i in range(runs + 1):
        t = time.perf_counter()
        ol.run_oracle(im, FLAGS, NITER, threads=threads)
        if i:
            times.append(time.perf_counter() - t)
    return statistics.median(times), "port", cores, "scalar C port with OpenMP, wall clock"


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    import jpegqs_b200 as qs
    im = qs.synth.make_image(WIDTH, HEIGHT, SUBSAMPLING, quality=QUALITY, seed=SEED)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    ol.ensure_built()
    kind = "reference" if ol.have_ref("avx512") else "port"
    times = []
    result = None
    cores = None
    nthreads = 0
    if kind == "reference":
        # untimed calibration: the reference defaults to all processors; on many-core hosts
        # fewer threads can be faster, so it gets the best of {all, 1/2, 1/4} (fair to it)
        lib = ol.reflib("avx512")
        allp = lib.qsref_num_procs()
        best = None
        for thr in sorted({allp, max(1, allp // 2), max(1, allp // 4)}, reverse=True):
            for rep in range(2):
                lib.qsref_take_log()
                ol.run_reference(im, FLAGS | (8 << 16), NITER, variant="avx512", threads=thr)
                log = lib.qsref_take_log().decode()
                ms = [float(l.split(":")[1].replace("ms", "")) for l in log.splitlines() if l.startswith("quantsmooth:")]
            if best is None or ms[-1] < best[0]:
                best = (ms[-1], thr)
        nthreads = best[1]
    for i in range(args.warmup + args.steps):
        if kind == "reference":
            lib = ol.reflib("avx512")
            cores = nthreads
            lib.qsref_take_log()
            result = ol.run_reference(im, FLAGS | (8 << 16), NITER, variant="avx512", threads=nthreads)
            log = lib.qsref_take_log().decode()
            ms = [float(l.split(":")[1].replace("ms", "")) for l in log.splitlines() if l.startswith("quantsmooth:")]
            dt = ms[-1] / 1e3
        else:
            cores = ol.oraclelib().qso_num_procs()
            t = time.perf_counter()
            result = ol.run_oracle(im, FLAGS, NITER, threads=0)
            dt = time.perf_counter() - t
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, result[0], [c.coef for c in result[1].comps])
    total = sum(times)
    mpix = WIDTH * HEIGHT / 1e6
    value = mpix * len(times) / total
    out = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "Mpixels/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(total / len(times) * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{WIDTH}x{HEIGHT} YCbCr 4:2:0, q=3 (flags 0), niter=3, whole image per step",
                   "timer": "reference's own 'quantsmooth: ms' line" if kind == "reference" else "wall clock"},
        "cpu_baseline": {"value": round(value, 3), "unit": "Mpixels/s", "cores": cores, "kind": kind,
                         "sample": "the full 8K image, every step"},
        "e2e": {"value": round(value, 3), "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result as .npy files")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import jpegqs_b200 as qs
    from jpegqs_b200 import multigpu as mg
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    ctx = qs.cuda.QsContext(local_rank)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                   # started early: nvidia-smi needs a moment before its first line
    ctx.set_profiling(True)

    im, mcu_rng, mcu_total = make_workload(world, rank)
    nblocks_rank = im.num_blocks
    total_blocks = nblocks_rank
    K, Wm = args.steps, args.warmup
    nbuf = K + Wm
    # a dedicated stream: the C ABI launches on it, the CUDA events below are recorded on it
    # and NCCL orders its halo exchange against it
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    mpix_job = WIDTH * HEIGHT * world / 1e6

    # ---- device-resident arm: a distinct pristine input buffer per step -----------------
    host_coefs = [torch.from_numpy(np.ascontiguousarray(c.coef)) for c in im.comps]
    dev_bufs = [[h.to(dev) for h in host_coefs] for _ in range(nbuf)]
    torch.cuda.synchronize()

    hblk_total, row0 = None, None
    link = None
    if world == 1:
        def step(i):
            ret, _ = ctx.run_device(im, [t.data_ptr() for t in dev_bufs[i]], [], FLAGS, NITER, stream)
            return ret
    else:
        # The C slab engine (include/jpegqs_cuda.h "one image sharded by MCU rows"): every rank
        # smooths its MCU rows; halo rows and out-of-range masks travel between the ranks inside
        # CUDA kernels through peer mailboxes (CUDA IPC over NVLink).  torch.distributed only
        # carries the IPC handles at start-up and the timing reductions.
        maxv = max(c.v_samp for c in im.comps)
        hblk_total = [-(-HEIGHT * world * c.v_samp // (8 * maxv)) for c in im.comps]
        row0 = [mg.comp_block_rows(mcu_rng, c.v_samp, ht)[0] for c, ht in zip(im.comps, hblk_total)]
        link = qs.cuda.QsLink(ctx, rank, world, max(c.wblk for c in im.comps))
        handles = [None] * world
        dist.all_gather_object(handles, link.export())
        link.connect_ipc(handles)

        def step(i):
            return ctx.run_slab(link, im, rank, world, row0, hblk_total, FLAGS, NITER,
                                coef_ptrs=[t.data_ptr() for t in dev_bufs[i]], up_ptrs=[], stream=stream)[0]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if rank == 0 and sampler.proc is not None:
        t_wait = time.perf_counter()
        while not sampler.lines and time.perf_counter() - t_wait < 10.0:
            time.sleep(0.05)
    for i in range(Wm):
        step(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    smooth_ms, smooth_n, idct_ms, idct_n = 0.0, 0, 0.0, 0
    barrier()
    sampler.t0 = time.perf_counter()
    e0.record()
    for i in range(K):
        ret = step(Wm + i)
        launches += ctx.last_launches
        a, b, c, d = ctx.kernel_stats()
        idct_ms += a; idct_n += b; smooth_ms += c; smooth_n += d
    e1.record()
    barrier()
    sampler.t1 = time.perf_counter()
    ms_total = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        nb = torch.tensor([nblocks_rank], dtype=torch.int64, device=dev)
        dist.all_reduce(nb)
        total_blocks = int(nb.item())
    ms_per_step = ms_total / K
    value = mpix_job / (ms_per_step / 1e3)

    # ---- e2e: the drop-in call itself --------------------------------------------------------
    # N=1: the library's exported do_quantsmooth(j_decompress_ptr, jvirt_barray_ptr*, jpegqs_control_t*)
    # (include/libjpegqs.h, reference libjpegqs.h:47-48) driven by a fake libjpeg front end whose
    # coefficient arrays are separately malloc'd, pageable block rows - what libjpeg's memory
    # manager hands over.  Only the call is timed (a libjpeg application has the arrays already,
    # reference quantsmooth.c:548-550); inside it: gather into pinned staging, H2D, kernels, D2H,
    # scatter back into the rows.
    e2e = None
    if not args.no_e2e:
        h2d = sum(c.coef.nbytes for c in im.comps)
        d2h = h2d
        if world == 1:
            import ctypes as C
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as ol                   # only its fake libjpeg front end (no smoothing code)
            ol.ensure_built()
            fn = C.cast(qs.cuda.load().do_quantsmooth, C.c_void_p)
            sessions = [ol.BoundarySession(im, scatter_rows=True) for _ in range(nbuf)]

            def e2e_step(i):
                ret = sessions[i].run(fn, FLAGS | 64, NITER)          # 64 = JPEGQS_TRANSCODE
                if ret != 0:
                    raise SystemExit(f"do_quantsmooth returned {ret}")
            api = ("do_quantsmooth(j_decompress_ptr, jvirt_barray_ptr*, jpegqs_control_t*) of libjpegqs_b200.so, "
                   "called through a fake libjpeg with scattered pageable block rows")
        else:
            pinned = []
            for _ in range(nbuf):
                row = []
                for c in im.comps:
                    p = qs.cuda.PinnedArray(c.coef.shape)
                    p.array[...] = c.coef
                    row.append(p)
                pinned.append(row)

            from jpegqs_b200.image import CoefImage, Component
            hosts = [CoefImage(im.width, im.height, im.colorspace,
                               [Component(pinned[i][k].array, c.quant.copy(), c.h_samp, c.v_samp, c.quant_tbl_no)
                                for k, c in enumerate(im.comps)]) for i in range(nbuf)]

            def e2e_step(i):
                ret = ctx.run_slab(link, hosts[i], rank, world, row0, hblk_total, FLAGS, NITER)[0]
                if ret != 0:
                    raise SystemExit(f"run_slab returned {ret}")
            api = ("jpegqs_cuda_run_slab (C slab engine) on every rank with caller-pinned host slabs: "
                   "H2D, kernels + kernel-side halo exchange over CUDA IPC mailboxes, D2H")

        for i in range(Wm):
            e2e_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            e2e_step(Wm + i)
        barrier()
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": round(mpix_job * K / dt, 2), "unit": "Mpixels/s", "h2d_bytes_per_step": h2d * world,
               "d2h_bytes_per_step": d2h * world, "ms_per_step": round(dt / K * 1e3, 3), "api": api}
        if world == 1:
            for sess in sessions:
                sess.close()
        else:
            for row in pinned:
                for p in row:
                    p.close()

    clocks = sampler.stop() if rank == 0 else None     # after the e2e phase: more samples under load

    # ---- roofline of the dominant kernel (smoothing pass) -------------------------------
    peak, peak_src = peaks()
    roofline = None
    if smooth_n:
        bytes_per_launch = ALGO_BYTES_PER_BLOCK_ITER * nblocks_rank
        avg_ms = smooth_ms / smooth_n
        achieved = bytes_per_launch / (avg_ms / 1e3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "smooth_traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        roofline = {"bound": "hbm", "kernel": "qs_smooth_kernel" + ("" if world == 1 else " (rank 0's slab)"),
                    "achieved": round(achieved, 2),
                    "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 5), "traffic": traffic,
                    "peak_source": peak_src, "avg_launch_ms": round(avg_ms, 4),
                    "algorithmic_bytes_per_launch": bytes_per_launch,
                    "share_of_step": round(smooth_ms / (ms_total if ms_total else 1), 4),
                    "note": "the path is FP32-issue bound, not HBM bound (SURVEY.md 8d, DESIGN.md 4); "
                            "see roofline_fp32"}
        # FP32-issue roofline.  Minimum FP32-pipe instructions of the order-exact arithmetic per
        # block-iteration, from the chunk schedule the kernel really runs for each component's quant
        # table: a coefficient has 56 horizontal (if not in column 0) + 32 border + 56 vertical (if not
        # in row 0) terms (+98 with DIAGONALS); 8 instructions per term, except in "uniform" chunks
        # (equal quant values) where the n coefficients share t and d*t: 3 + 5n per term.
        def min_fp_per_block(quant, diag):
            total = 0
            for typ, _first, idx in qs.cuda.chunk_schedule(quant):
                if typ == 2:
                    total += (144 + (98 if diag else 0)) * (3 + 5 * len(idx))
                else:                                  # plain, edge and mixed chunks: 8 per term
                    for i in idx:
                        terms = 32 + (56 if i & 7 else 0) + (56 if i > 7 else 0) + (98 if diag else 0)
                        total += 8 * terms
            return total
        fp_inst = sum(min_fp_per_block(c.quant, bool(FLAGS & 1)) * c.wblk * c.hblk for c in im.comps) / 32.0
        fp_inst_plain = 8288 * 8 * nblocks_rank / 32.0                  # without the uniform-chunk sharing
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        issue_peak = 148 * 4 * sm_mhz * 1e6                            # warp-instr/s at 1 per SMSP per clock
        roofline_fp32 = {"bound": "fp32-issue", "achieved": round(fp_inst / (avg_ms / 1e3) / 1e12, 4),
                         "peak": round(issue_peak / 1e12, 4), "unit": "T warp-instr/s",
                         "frac": round(fp_inst / (avg_ms / 1e3) / issue_peak, 4),
                         "frac_counting_8_per_term": round(fp_inst_plain / (avg_ms / 1e3) / issue_peak, 4),
                         "note": "minimum FP32-pipe instructions of the order-exact arithmetic for the chunk schedules in "
                                 "use (uniform chunks: 3 + 5n per term) / (148 SM x 4 sub-partitions x measured SM clock); "
                                 "frac_counting_8_per_term is round 1's figure (8 per term everywhere)"}
    else:
        roofline_fp32 = None

    # ---- CPU baseline beside it (rank 0, N=1 only) ---------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sec, kind, cores, how = cpu_reference_time(im, threads=0, runs=5)
        cpu = {"value": round(WIDTH * HEIGHT / 1e6 / sec, 3), "unit": "Mpixels/s", "cores": cores, "kind": kind,
               "sample": f"the full 8K image, 1 warm-up + median of 5 runs ({how})"}

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ret, [t.cpu().numpy() for t in dev_bufs[Wm + K - 1]],
                     prefix="" if world == 1 else f"rank{rank}_", world=world)

    if rank == 0:
        out = {
            "metric": METRIC, "value": round(value, 2), "unit": "Mpixels/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{WIDTH}x{HEIGHT * world} YCbCr 4:2:0 (8K x{world} stacked), q=3 (flags 0), "
                                   f"niter=3, quality-50 Annex-K tables, seed {SEED}",
                       "blocks": total_blocks,
                       "cache": "a distinct pristine input buffer per step (100 MB each, "
                                f"{nbuf} buffers > 126 MB L2)",
                       "sharding": "none" if world == 1 else
                       f"MCU rows over {world} GPUs (one process each); halo rows + out-of-range masks exchanged by "
                       "CUDA kernels through peer mailboxes (CUDA IPC / NVLink), no host sync, no NCCL on the data path"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "roofline_fp32": roofline_fp32, "cpu_baseline": cpu,
            "kernel_ms_per_step": {"idct_pass": round(idct_ms / K, 4), "smooth_pass": round(smooth_ms / K, 4)},
        }
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
