"""The `jpegqs` command line tool (csrc/jpegqs.c) and its JPEG coefficient codec
(csrc/jpegcoef.c).  CPU leg: the codec is a lossless transcoder (`-n 0` never reaches the
CUDA back end) on baseline / progressive / sub-sampled / restart-marker / grayscale files
written by Pillow's libjpeg-turbo, and markers are copied per `-c`.  GPU leg: the CUDA-backed
tool must write byte-identical files to oracle/_ref/jpegqs_ref (the same front end linked
against the UNMODIFIED reference do_quantsmooth, built by oracle/Makefile); the digests of that
tool's files are stored in tests/golden/reference_outputs.json (see reference_outputs())."""
import os
import subprocess

import numpy as np
import pytest

from golden_io import file_digest, reference_output

PIL = pytest.importorskip("PIL.Image")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "jpeg-quantsmooth_b200", "csrc", "jpegqs")
REF_EXE = os.path.join(ROOT, "oracle", "_ref", "jpegqs_ref")


def _picture(w, h, gray, seed):
    rng = np.random.RandomState(seed)
    y, x = np.mgrid[0:h, 0:w]
    a = (128 + 60 * np.sin(x / 17.0) + 50 * np.cos(y / 23.0) + rng.randint(-20, 20, (h, w))).clip(0, 255).astype(np.uint8)
    if gray:
        return PIL.fromarray(a, "L")
    b = (128 + 60 * np.cos(x / 11.0) + rng.randint(-30, 30, (h, w))).clip(0, 255).astype(np.uint8)
    c = (128 + 80 * np.sin((x + y) / 29.0)).clip(0, 255).astype(np.uint8)
    return PIL.fromarray(np.stack([a, b, c], -1), "RGB")


FILES = [
    ("base420", 64, 48, False, dict(quality=75)),
    ("base444", 123, 77, False, dict(quality=90, subsampling=0)),
    ("prog420", 200, 133, False, dict(quality=50, subsampling=2, progressive=True)),
    ("gray", 97, 61, True, dict(quality=85)),
    ("opt422", 160, 120, False, dict(quality=30, subsampling=1, optimize=True)),
    ("prog444", 333, 211, False, dict(quality=95, progressive=True, subsampling=0)),
    ("rst", 250, 190, False, dict(quality=80, restart_marker_rows=1)),
    ("progrst", 250, 190, False, dict(quality=80, progressive=True, restart_marker_blocks=7)),
    ("tinyprog", 17, 9, True, dict(quality=60, progressive=True)),
    # dense blocks with large magnitudes (long codes, the two-step decode path, FF bytes to stuff) and
    # nearly empty ones (long zero runs, ZRL): the two ends of the block coder's fast paths
    ("dense444", 320, 200, False, dict(quality=100, subsampling=0)),
    ("coarse420", 300, 220, False, dict(quality=3)),
]


def make_jpegs(d):
    out = {}
    for k, (name, w, h, gray, kw) in enumerate(FILES):
        p = os.path.join(d, name + ".jpg")
        _picture(w, h, gray, k).save(p, comment=b"made by the test suite", **kw)
        out[name] = p
    return out


@pytest.fixture(scope="module")
def jpegs(tmp_path_factory):
    return make_jpegs(str(tmp_path_factory.mktemp("jpegs")))


def check_input(name, path):
    """The stored outputs of the reference were made from these very files."""
    assert file_digest(path) == reference_output(f"input/{name}"), \
        f"{name}: this Pillow writes other bytes than the one the reference outputs were made with"


def _pixels(path):
    im = PIL.open(path)
    return np.asarray(im if im.mode == "L" else im.convert("RGB"))


def _markers(path):
    data = open(path, "rb").read()
    i, found = 2, []
    while i + 4 <= len(data) and data[i] == 0xFF:
        code = data[i + 1]
        if code == 0xDA:
            break
        n = int.from_bytes(data[i + 2:i + 4], "big")
        found.append((code, data[i + 4:i + 2 + n]))
        i += 2 + n
    return found


def test_tool_is_built():
    assert os.path.exists(EXE), "build() must produce csrc/jpegqs"


@pytest.mark.parametrize("name", [f[0] for f in FILES])
@pytest.mark.parametrize("optimize", [False, True])
def test_codec_is_a_lossless_transcoder(jpegs, tmp_path, name, optimize):
    out = str(tmp_path / "out.jpg")
    r = subprocess.run([EXE, "-n", "0", "-i", "0"] + (["-o"] if optimize else []) + [jpegs[name], out],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(_pixels(jpegs[name]), _pixels(out))
    # re-reading our own output must be lossless as well
    out2 = str(tmp_path / "out2.jpg")
    assert subprocess.run([EXE, "-n", "0", "-i", "0", out, out2]).returncode == 0
    assert np.array_equal(_pixels(out), _pixels(out2))


def test_writer_bytes_do_not_depend_on_the_thread_count(jpegs, tmp_path):
    """The writer codes segments of MCU rows on worker threads and splices their bits: the file
    must be byte for byte the sequential coder's (1 thread), also with -o and odd thread counts."""
    for name in ("base420", "prog420", "gray", "rst", "base444", "dense444", "coarse420"):
        if name not in jpegs:
            continue
        for optimize in ([], ["-o"]):
            want = None
            for threads in ("1", "2", "3", "7", "64"):
                out = str(tmp_path / f"t{threads}.jpg")
                env = dict(os.environ, JPEGQS_CODEC_THREADS=threads)
                assert subprocess.run([EXE, "-n", "0", "-i", "0"] + optimize + [jpegs[name], out], env=env).returncode == 0
                got = open(out, "rb").read()
                if want is None:
                    want = got
                assert got == want, (name, optimize, threads)
            out = str(tmp_path / "tflag.jpg")             # the -t option, environment unset
            env = {k: v for k, v in os.environ.items() if k != "JPEGQS_CODEC_THREADS"}
            assert subprocess.run([EXE, "-n", "0", "-i", "0", "-t", "5"] + optimize + [jpegs[name], out], env=env).returncode == 0
            assert open(out, "rb").read() == want


def _big_picture(w, h, seed, **kw):
    rng = np.random.RandomState(seed)
    y, x = np.mgrid[0:h, 0:w]
    a = np.stack([128 + 70 * np.sin(x / 31.0) + 40 * np.cos(y / 19.0), 128 + 60 * np.cos((x + y) / 47.0),
                  128 + 80 * np.sin((x - y) / 23.0)], -1) + rng.normal(0, 9, (h, w, 3))
    return PIL.fromarray(a.clip(0, 255).astype(np.uint8), "RGB")


@pytest.mark.parametrize("name", ["base420", "base444", "gray", "opt422", "rst", "dense444", "coarse420", "big420", "big444rst",
                                  "biggray", "big422opt", "bigcmyk"])
def test_threaded_decoder_equals_the_serial_one(jpegs, tmp_path, name):
    """Sequential scans are decoded on several threads (speculative parsing of chunks, stitched at
    the points where they synchronize; restart intervals as they are).  The result must be the
    one-thread decoder's for every chunk and thread count; the trace says which path ran."""
    big = {"big420": (1400, 900, dict(quality=85)), "big444rst": (900, 700, dict(quality=92, subsampling=0, restart_marker_rows=2)),
           "biggray": (1100, 800, dict(quality=70)), "big422opt": (1000, 640, dict(quality=60, subsampling=1, optimize=True))}
    big["bigcmyk"] = (640, 480, dict(quality=85))       # one Huffman table pair for all four components: stays on one thread
    if name in big:
        w, h, kw = big[name]
        src = str(tmp_path / (name + ".jpg"))
        im = _big_picture(w, h, len(name))
        if name == "biggray":
            im = im.convert("L")
        if name == "bigcmyk":
            im = PIL.fromarray(np.dstack([np.asarray(im), np.asarray(im)[:, ::-1, 0]]), "CMYK")
        im.save(src, **kw)
    else:
        src = jpegs[name]
    ref = str(tmp_path / "serial.jpg")
    env = dict(os.environ, JPEGQS_SERIAL_DECODE="1")
    assert subprocess.run([EXE, "-n", "0", "-i", "0", src, ref], env=env).returncode == 0
    want = open(ref, "rb").read()
    for threads, min_bytes in (("4", "300"), ("7", "300"), ("16", "2000"), ("5", None)):
        out = str(tmp_path / f"t{threads}.jpg")
        env = dict(os.environ, JPEGQS_CODEC_THREADS=threads, JPEGQS_CODEC_TRACE="1")
        if min_bytes:
            env["JPEGQS_PAR_MIN_BYTES"] = min_bytes
        r = subprocess.run([EXE, "-n", "0", "-i", "0", src, out], env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert open(out, "rb").read() == want, (name, threads)
        if name == "bigcmyk":
            assert "decoded on" not in r.stderr, r.stderr
        elif name in big and min_bytes:      # (with the default threshold only segments of 128 KB and more take the threaded path)
            assert "decoded on" in r.stderr and "abandoned" not in r.stderr, r.stderr
            if "rst" in name:
                assert "restart intervals" in r.stderr


def test_marker_copy_levels(jpegs, tmp_path):
    """-c selects the COPIED markers; the JFIF APP0 is not one of them: libjpeg writes it itself
    for every grayscale / YCbCr output (jcmarker.c write_file_header) with the source's version
    and density (jctrans.c jpeg_copy_critical_parameters), and so does this codec."""
    src = str(tmp_path / "src.jpg")
    _picture(64, 48, False, 3).save(src, quality=75, comment=b"made by the test suite", dpi=(300, 150),
                                    exif=b"Exif\x00\x00II*\x00\x08\x00\x00\x00\x00\x00\x00\x00\x00\x00")
    for level, want_com, want_app in ((2, True, True), (1, True, False), (0, False, False)):
        out = str(tmp_path / f"c{level}.jpg")
        assert subprocess.run([EXE, "-n", "0", "-i", "0", "-c", str(level), src, out]).returncode == 0
        m = _markers(out)
        assert any(c == 0xFE and b"made by the test suite" in d for c, d in m) == want_com
        jfif = [d for c, d in m if c == 0xE0 and d[:5] == b"JFIF\x00"]
        assert len(jfif) == 1 and m[0][0] == 0xE0                      # once, first, at every level
        assert jfif[0][7] == 1 and jfif[0][8:12] == (300).to_bytes(2, "big") + (150).to_bytes(2, "big")
        assert any(c == 0xE1 and d[:4] == b"Exif" for c, d in m) == want_app
        assert PIL.open(out).info.get("dpi") == (300, 150)


@pytest.mark.parametrize("mode", ["CMYK", "RGB"])
def test_adobe_marker_keeps_the_colour_transform(tmp_path, mode):
    """RGB / CMYK / YCCK files carry their colour transform in the Adobe APP14 marker; libjpeg
    writes it for every such output whatever -c says.  Without it a decoder guesses YCbCr / CMYK
    and shows wrong colours (ADVICE round 1)."""
    src = str(tmp_path / "src.jpg")
    pic = _picture(80, 56, False, 5)
    if mode == "CMYK":
        pic.convert("CMYK").save(src, quality=85)
    else:
        try:
            pic.save(src, quality=85, keep_rgb=True)                     # Pillow >= 10.2: JCS_RGB, no transform
        except TypeError:
            pytest.skip("this Pillow cannot write untransformed RGB JPEGs")
    want = np.asarray(PIL.open(src).convert("RGB"))
    for level in (0, 2):
        out = str(tmp_path / f"o{level}.jpg")
        assert subprocess.run([EXE, "-n", "0", "-i", "0", "-c", str(level), src, out]).returncode == 0
        adobe = [d for c, d in _markers(out) if c == 0xEE and d[:5] == b"Adobe"]
        assert len(adobe) == 1 and not any(c == 0xE0 for c, _ in _markers(out))
        assert np.array_equal(np.asarray(PIL.open(out).convert("RGB")), want)


def test_exit_status_follows_the_reference(jpegs, tmp_path):
    """quantsmooth.c:626: 2 when the codec met recoverable damage (libjpeg warnings), else 0;
    an unwritable output is 1 (round 1 returned 0 for it)."""
    data = open(jpegs["base420"], "rb").read()
    cut = tmp_path / "cut.jpg"
    cut.write_bytes(data[:len(data) * 2 // 3])                            # truncated: no EOI
    r = subprocess.run([EXE, "-n", "0", "-i", "0", str(cut), str(tmp_path / "o.jpg")], capture_output=True)
    assert r.returncode == 2 and (tmp_path / "o.jpg").exists()
    if os.path.exists("/dev/full"):
        r = subprocess.run([EXE, "-n", "0", "-i", "0", jpegs["base420"], "/dev/full"], capture_output=True)
        assert r.returncode == 1


def test_batch_mode_equals_single_runs(jpegs, tmp_path):
    """--batch: several "input output" pairs in one process (CUDA start-up paid once)."""
    names = ["base420", "prog420", "gray"]
    args = [EXE, "-n", "0", "-i", "0", "--batch"]
    for n in names:
        args += [jpegs[n], str(tmp_path / f"b_{n}.jpg")]
    assert subprocess.run(args).returncode == 0
    for n in names:
        single = str(tmp_path / f"s_{n}.jpg")
        assert subprocess.run([EXE, "-n", "0", "-i", "0", jpegs[n], single]).returncode == 0
        assert open(single, "rb").read() == open(tmp_path / f"b_{n}.jpg", "rb").read()
    assert subprocess.run([EXE, "--batch", jpegs["gray"]], capture_output=True).returncode == 1     # odd count: usage


def test_batch_pipeline_keeps_the_order_of_dependent_pairs(jpegs, tmp_path):
    """--batch runs read / smooth / write as a three-stage pipeline.  A pair whose input is the
    output of an earlier pair must see the finished file, a failing pair must not disturb the
    others, and the files must be those of the one-pair-after-the-other mode (JPEGQS_NO_PIPELINE)."""
    def run(tag, env):
        a, b, c, d, e = (str(tmp_path / f"{tag}_{k}.jpg") for k in "abcde")
        args = [EXE, "-n", "0", "-i", "0", "-t", "3", "--batch",
                jpegs["base444"], a,              # a
                a, b,                             # reads what the first pair writes
                str(tmp_path / "missing.jpg"), str(tmp_path / f"{tag}_x.jpg"),
                jpegs["prog420"], c,
                jpegs["dense444"], d,
                d, d,                             # in place, after the pair before it
                jpegs["gray"], e, jpegs["base420"], e]     # the same output twice: the later pair's stays
        r = subprocess.run(args, capture_output=True, text=True, env=env)
        assert r.returncode == 1 and "missing.jpg" in r.stderr
        assert not os.path.exists(tmp_path / f"{tag}_x.jpg")
        return [open(f, "rb").read() for f in (a, b, c, d, e)]
    piped = run("p", dict(os.environ))
    plain = run("s", dict(os.environ, JPEGQS_NO_PIPELINE="1"))
    assert piped == plain
    assert piped[0] == piped[1]                   # transcoding our own output changes nothing
    single = str(tmp_path / "single.jpg")
    assert subprocess.run([EXE, "-n", "0", "-i", "0", "-t", "3", jpegs["base420"], single]).returncode == 0
    assert piped[4] == open(single, "rb").read()


def test_bad_input_and_usage(tmp_path):
    bad = tmp_path / "bad.jpg"
    bad.write_bytes(b"this is not a jpeg")
    r = subprocess.run([EXE, "-n", "0", str(bad), str(tmp_path / "o.jpg")], capture_output=True, text=True)
    assert r.returncode == 1 and "not a JPEG" in r.stderr
    assert subprocess.run([EXE], capture_output=True).returncode == 1
    assert subprocess.run([EXE, "-q", "x", "a", "b"], capture_output=True).returncode == 1


def test_no_cpu_fallback_in_the_tool(jpegs, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    out = tmp_path / "o.jpg"
    r = subprocess.run([EXE, "-q", "3", jpegs["base420"], str(out)], capture_output=True, text=True)
    assert r.returncode == 2 and "CUDA back end unavailable" in r.stderr
    assert not out.exists()


REF_TOOL_CASES = [
    ("base420", ["-q", "3"]), ("base420", ["-q", "6", "-n", "2"]), ("prog420", ["-q", "4", "-n", "2", "-o"]),
    ("base444", ["-q", "5", "-n", "2"]), ("gray", ["-q", "3", "-n", "4"]), ("opt422", ["-q", "6"]),
    ("prog444", ["-q", "1", "-n", "2"]), ("rst", ["-q", "0"]), ("progrst", ["-q", "1", "-o"]),
    ("opt422", ["-q", "2", "-o"]),
    ("tinyprog", ["-q", "3"]), ("base420", ["-f", "16", "-n", "2"]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,args", REF_TOOL_CASES)
def test_cuda_tool_writes_the_reference_tools_bytes(jpegs, tmp_path, name, args):
    # UPSAMPLE_UV cases use widths that are multiples of the MCU: for other widths the reference
    # reads uninitialised memory when it pads the up-sampled plane (DESIGN.md "reference quirks")
    check_input(name, jpegs[name])
    a = str(tmp_path / "cuda.jpg")
    r1 = subprocess.run([EXE, "-i", "0"] + args + [jpegs[name], a], capture_output=True, text=True)
    assert r1.returncode == 0, r1.stderr
    assert file_digest(a) == reference_output(f"jpegqs_ref/{name} {' '.join(args)}")
    PIL.open(a).load()                      # and it is a decodable JPEG


@pytest.mark.gpu
@pytest.mark.parametrize("name", [f[0] for f in FILES])
def test_device_decode_equals_libjpeg_turbo(jpegs, tmp_path, name):
    """--ppm with -n 0 is a plain decoder: islow IDCT + fancy up-sampling + YCbCr->RGB on the
    device must reproduce Pillow's libjpeg-turbo decode of the same file exactly."""
    out = str(tmp_path / "o.ppm")
    r = subprocess.run([EXE, "-n", "0", "-i", "0", "--ppm", jpegs[name], out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = np.asarray(PIL.open(out))
    want = np.asarray(PIL.open(jpegs[name]))
    assert got.shape == want.shape
    assert np.array_equal(got, want), f"max diff {np.abs(got.astype(int) - want.astype(int)).max()}"


@pytest.mark.gpu
@pytest.mark.parametrize("name,args", [("base420", ["-q", "3"]), ("prog420", ["-q", "6"]), ("gray", ["-q", "4"]),
                                       ("opt422", ["-q", "5", "-n", "2"])])
def test_smoothed_pixels_equal_decoding_the_smoothed_file(jpegs, tmp_path, name, args):
    """jpegqs_start_decompress semantics (quantsmooth.h:2880-2904): the pixels libjpeg would
    deliver for the smoothed coefficients = decoding the transcoded file."""
    ppm, jpg = str(tmp_path / "o.ppm"), str(tmp_path / "o.jpg")
    assert subprocess.run([EXE, "-i", "0"] + args + ["--ppm", jpegs[name], ppm]).returncode == 0
    assert subprocess.run([EXE, "-i", "0"] + args + [jpegs[name], jpg]).returncode == 0
    assert np.array_equal(np.asarray(PIL.open(ppm)), np.asarray(PIL.open(jpg)))


@pytest.mark.gpu
def test_batch_pipeline_on_the_device(jpegs, tmp_path):
    """--batch with real smoothing: the reader and writer threads work on other pairs while the
    calling thread runs do_quantsmooth; every file equals the one a single-pair process writes."""
    names = ["base420", "prog444", "gray", "dense444", "opt422", "rst"]
    args = [EXE, "-q", "3", "-i", "0", "--batch"]
    for n in names:
        args += [jpegs[n], str(tmp_path / f"b_{n}.jpg")]
    r = subprocess.run(args, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for n in names:
        single = str(tmp_path / f"s_{n}.jpg")
        assert subprocess.run([EXE, "-q", "3", "-i", "0", jpegs[n], single]).returncode == 0
        assert open(single, "rb").read() == open(tmp_path / f"b_{n}.jpg", "rb").read(), n


def test_codec_survives_corrupt_input(jpegs, tmp_path):
    """Mutated / truncated files must be rejected or decoded, never crash: the codec is built
    with AddressSanitizer + UBSan (do_quantsmooth stubbed out) and fed 300 seeded mutations."""
    exe = str(tmp_path / "jq_asan")
    stub = tmp_path / "stub.c"
    stub.write_text('#include <jpeglib.h>\n#include "libjpegqs.h"\n'
                    "int do_quantsmooth(j_decompress_ptr a, jvirt_barray_ptr *b, jpegqs_control_t *c)"
                    " { (void)a; (void)b; (void)c; return 0; }\n")
    csrc = os.path.join(ROOT, "jpeg-quantsmooth_b200", "csrc")
    r = subprocess.run(["/usr/bin/gcc", "-O1", "-g", "-fsanitize=address,undefined", "-DJPEGQS_NO_CUDA_RENDER",
                        "-I", os.path.join(ROOT, "include", "libjpeg62"), "-I", os.path.join(ROOT, "include"), "-I", csrc,
                        "-o", exe, os.path.join(csrc, "jpegqs.c"), os.path.join(csrc, "jpegcoef.c"), str(stub), "-lpthread"],
                       capture_output=True, text=True)
    if r.returncode:
        pytest.skip("sanitizer build unavailable: " + r.stderr[-200:])
    rng = np.random.RandomState(7)
    seeds = [open(jpegs[n], "rb").read() for n in ("base420", "prog420", "gray", "rst", "tinyprog", "base444", "opt422")]
    for it in range(300):
        d = bytearray(seeds[it % len(seeds)])
        mode = rng.randint(4)
        if mode == 0:
            for _ in range(rng.randint(1, 6)):
                d[rng.randint(len(d))] = rng.randint(256)
        elif mode == 1:
            d = d[:rng.randint(2, len(d))]
        elif mode == 2:
            i = rng.randint(2, len(d) - 4)
            d[i:i + 4] = bytes(rng.randint(0, 256, 4).tolist())
        else:
            i = rng.randint(len(d))
            d = d[:i] + bytes(rng.randint(0, 256, rng.randint(1, 40)).tolist()) + d[i:]
        f = tmp_path / "f.jpg"
        f.write_bytes(bytes(d))
        out = tmp_path / "o.jpg"
        if out.exists():
            out.unlink()
        env = dict(os.environ, JPEGQS_SERIAL_DECODE="1")
        r = subprocess.run([exe, "-n", "0", "-i", "0", str(f), str(out)], capture_output=True, timeout=60, env=env)
        # 0 decoded, 1 rejected, 2 decoded with recoverable damage (the reference's warning status)
        assert r.returncode in (0, 1, 2), (it, r.returncode, r.stderr.decode()[-800:])
        # the threaded decoder (forced onto these small files) must give up or agree: same status, same bytes
        want = out.read_bytes() if out.exists() else None
        if out.exists():
            out.unlink()
        env = dict(os.environ, JPEGQS_PAR_MIN_BYTES="200", JPEGQS_CODEC_THREADS=str(4 + it % 5))
        r2 = subprocess.run([exe, "-n", "0", "-i", "0", str(f), str(out)], capture_output=True, timeout=60, env=env)
        assert r2.returncode == r.returncode, (it, r.returncode, r2.returncode, r2.stderr.decode()[-800:])
        assert (out.read_bytes() if out.exists() else None) == want, it


def reference_outputs(tmpdir):
    """The inputs' digests and oracle/_ref/jpegqs_ref's files for the cases above."""
    jpegs = make_jpegs(tmpdir)
    out = {f"input/{name}": file_digest(p) for name, p in jpegs.items()}
    for name, args in REF_TOOL_CASES:
        b = os.path.join(tmpdir, "ref.jpg")
        subprocess.run([REF_EXE, "-i", "0"] + args + [jpegs[name], b], check=True, capture_output=True)
        out[f"jpegqs_ref/{name} {' '.join(args)}"] = file_digest(b)
    return out
