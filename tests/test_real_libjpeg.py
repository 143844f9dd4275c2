"""The libjpeg-facing half meets a REAL libjpeg: Pillow's wheel carries libjpeg-turbo 3.1
(libjpeg API/ABI 6.2, no headers); include/libjpeg62/jpeglib.h declares that API by hand and the
shipped library is compiled against it.

CPU leg: the hand-declared structs are accepted by the real library (its own struct-size /
version check) and a real decode through them gives the coefficients csrc/jpegcoef.c reads;
the reference's CLI on real libjpeg writes the very bytes this repository's codec writes.
GPU leg: the reference's OWN callers run on the CUDA back end with real libjpeg -
oracle/_ref/refcli_b200 is the unmodified reference quantsmooth.c whose SIMD dispatcher links
the tier workers exported by libjpegqs_b200.so; example_b200 is the reference's example.c
(jpegqs_start_decompress -> jpeg_read_scanlines) - and must reproduce the all-CPU builds of the
same sources (refcli_cpu / example_cpu) byte for byte.  What the all-CPU builds write is stored in
tests/golden/reference_outputs.json (see reference_outputs())."""
import glob
import json
import os
import subprocess

import numpy as np
import pytest

PIL = pytest.importorskip("PIL.Image")
import PIL as _PIL  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "jpeg-quantsmooth_b200", "csrc")
REFDIR = os.path.join(ROOT, "oracle", "_ref")
_so = sorted(glob.glob(os.path.join(os.path.dirname(os.path.realpath(_PIL.__file__)), "..", "pillow.libs", "libjpeg*.so*")))
JPEG_SO = os.path.realpath(_so[0]) if _so else None
pytestmark = pytest.mark.skipif(JPEG_SO is None, reason="no libjpeg shared library inside Pillow")

from golden_io import digest, file_digest, reference_output  # noqa: E402
from test_cli import _picture, check_input, make_jpegs  # noqa: E402


def make_real_jpegs(d):
    out = make_jpegs(d)
    # sizes that are multiples of the MCU: the reference's UPSAMPLE_UV reads uninitialised memory
    # otherwise (DESIGN.md "reference quirks"), so q6 is compared on these only
    for name, w, h, kw in (("mcu420", 192, 144, dict(quality=60)), ("mcuprog", 256, 160, dict(quality=85, progressive=True)),
                           ("mcu422", 160, 96, dict(quality=40, subsampling=1))):
        p = os.path.join(d, name + ".jpg")
        _picture(w, h, False, 11).save(p, **kw)
        out[name] = p
    return out


@pytest.fixture(scope="module")
def jpegs(tmp_path_factory):
    return make_real_jpegs(str(tmp_path_factory.mktemp("real")))


DUMP = r'''
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <jpeglib.h>
#ifdef USE_JQ
#include "jpegcoef.h"
#endif
static void dump(struct jpeg_decompress_struct *ci, jvirt_barray_ptr *arr) {
	int c;
	printf("%ux%u %d cs%d\n", ci->image_width, ci->image_height, ci->num_components, (int)ci->jpeg_color_space);
	for (c = 0; c < ci->num_components; c++) {
		jpeg_component_info *k = &ci->comp_info[c]; unsigned long h = 1469598103934665603ul; JDIMENSION y, x; int i;
		for (y = 0; y < k->height_in_blocks; y++) {
			JBLOCKARRAY r = ci->mem->access_virt_barray((j_common_ptr)ci, arr[c], y, 1, FALSE);
			for (x = 0; x < k->width_in_blocks; x++) for (i = 0; i < 64; i++) h = (h ^ (unsigned short)r[0][x][i]) * 1099511628211ul;
		}
		for (i = 0; i < 64; i++) h = (h ^ k->quant_table->quantval[i]) * 1099511628211ul;
		printf("%d: %dx%d t%d %ux%u %lx\n", c, k->h_samp_factor, k->v_samp_factor, k->quant_tbl_no, k->width_in_blocks, k->height_in_blocks, h);
	}
}
int main(int argc, char **argv) {
	(void)argc;
#ifdef USE_JQ
	FILE *f = fopen(argv[1], "rb"); static unsigned char buf[1 << 22]; size_t n = fread(buf, 1, sizeof(buf), f);
	jq_image im; char err[256];
	if (jq_read(buf, n, 2, &im, err)) { puts(err); return 1; }
	dump(&im.cinfo, im.coef_arrays);
#else
	struct jpeg_decompress_struct ci; struct jpeg_error_mgr err; FILE *f = fopen(argv[1], "rb");
	ci.err = jpeg_std_error(&err);
	jpeg_create_decompress(&ci);          /* the real library checks sizeof(ci) and the version here */
	jpeg_stdio_src(&ci, f);
	jpeg_read_header(&ci, TRUE);
	dump(&ci, jpeg_read_coefficients(&ci));
	{ struct jpeg_compress_struct co; co.err = jpeg_std_error(&err); jpeg_create_compress(&co); jpeg_destroy_compress(&co); }
#endif
	return 0;
}
'''


def test_declared_abi_is_the_real_librarys_and_both_codecs_agree(jpegs, tmp_path):
    src = tmp_path / "dump.c"
    src.write_text(DUMP)
    inc = ["-I", os.path.join(ROOT, "include", "libjpeg62"), "-I", os.path.join(ROOT, "include"), "-I", CSRC]
    real, ours = str(tmp_path / "dump_real"), str(tmp_path / "dump_jq")
    subprocess.run(["/usr/bin/gcc", "-O1"] + inc + [str(src), "-o", real, JPEG_SO, f"-Wl,-rpath,{os.path.dirname(JPEG_SO)}"], check=True)
    subprocess.run(["/usr/bin/gcc", "-O1", "-DUSE_JQ"] + inc + [str(src), os.path.join(CSRC, "jpegcoef.c"), "-o", ours, "-lpthread"], check=True)
    for name, path in jpegs.items():
        a = subprocess.run([real, path], capture_output=True, text=True)
        b = subprocess.run([ours, path], capture_output=True, text=True)
        assert a.returncode == 0 and b.returncode == 0, (name, a.stderr, b.stdout)
        assert a.stdout == b.stdout, name


def _have(*names):
    return all(os.path.exists(os.path.join(REFDIR, n)) for n in names)


def _b200_env():
    """refcli_b200 / example_b200 load libjpegqs_b200.so from this tree's csrc/, named explicitly:
    their run path only finds it while oracle/_ref sits inside the tree it was built in."""
    path = os.environ.get("LD_LIBRARY_PATH")
    return dict(os.environ, LD_LIBRARY_PATH=CSRC + (os.pathsep + path if path else ""))


REFCLI_CASES = [(name, args) for name in ("base420", "gray", "prog420", "opt422", "rst")
                for args in (["-q", "3", "-n", "2"], ["-q", "4", "-n", "1", "-o"], ["-q", "2"])]


@pytest.mark.skipif(not _have("jpegqs_ref"), reason="oracle/_ref not built")
def test_reference_cli_on_real_libjpeg_writes_this_codecs_bytes(jpegs, tmp_path):
    """quantsmooth.c + libjpeg-turbo (refcli_cpu, stored) vs the same smoothing behind
    csrc/jpegcoef.c + jpegqs.c: the files are byte-identical, i.e. the codec reproduces
    jpeg_copy_critical_parameters + jpeg_write_coefficients + jcopy_markers (JFIF / Adobe handling
    included)."""
    for name, args in REFCLI_CASES:
        check_input(name, jpegs[name])
        b = str(tmp_path / "jq.jpg")
        r2 = subprocess.run([os.path.join(REFDIR, "jpegqs_ref"), "-i", "0"] + args + [jpegs[name], b], capture_output=True)
        assert r2.returncode == 0
        assert file_digest(b) == reference_output(f"refcli_cpu/{name} {' '.join(args)}"), (name, args)


def test_random_files_one_thread_threaded_and_libjpeg_turbo_agree(tmp_path):
    """A short run of tools/codec_difftest.py: random size / quality / sub-sampling / optimised tables /
    restart intervals / progressive files; the lossless transcode must give libjpeg-turbo's bytes (as
    refcli_cpu wrote them, stored) with the one-thread reader and with the threaded reader (random thread
    count and chunk size)."""
    digests = tmp_path / "refcli_cpu.json"
    digests.write_text(json.dumps(reference_output("codec_difftest/77 30")))
    r = subprocess.run([os.sys.executable, os.path.join(ROOT, "tools", "codec_difftest.py"), "77", "30", str(digests)],
                       cwd=str(tmp_path), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "done 30 bad 0" in r.stdout, r.stdout[-2000:]


B200_CLI_CASES = {"-q 3": ("base420", "prog420", "gray", "rst"), "-q 4 -n 2": ("prog420", "opt422", "base444"),
                  "-q 5 -n 2": ("base420", "mcu420", "base444"), "-q 6": ("mcu420", "mcuprog", "mcu422"),
                  "-q 1": ("gray", "opt422", "rst"), "-q 3 -o": ("base420", "prog420", "opt422")}


@pytest.mark.gpu
@pytest.mark.skipif(not _have("refcli_b200"), reason="oracle/_ref not built")
@pytest.mark.parametrize("args", [["-q", "3"], ["-q", "4", "-n", "2"], ["-q", "5", "-n", "2"], ["-q", "6"], ["-q", "1"], ["-q", "3", "-o"]])
def test_unmodified_reference_cli_runs_on_the_cuda_back_end(jpegs, tmp_path, args):
    # each file costs a fresh process with its CUDA start-up: the flavours are spread over the argument sets
    # (q6 on MCU-multiple sizes only, see the fixture)
    for name in B200_CLI_CASES[" ".join(args)]:
        check_input(name, jpegs[name])
        b = str(tmp_path / "b200.jpg")
        r2 = subprocess.run([os.path.join(REFDIR, "refcli_b200"), "-i", "16"] + args + [jpegs[name], b],
                            capture_output=True, text=True, env=_b200_env())
        assert r2.returncode == 0, r2.stderr
        assert "CUDA sm_100a" in r2.stderr, r2.stderr            # it really went through the tier slot into the GPU
        assert file_digest(b) == reference_output(f"refcli_cpu/{name} {' '.join(args)}"), (name, args)


def _rgb_digest(path):
    a = np.asarray(PIL.open(path).convert("RGB"))
    return digest(np.array(a.shape), a)


EXAMPLE_FILES = ("mcu420", "mcuprog", "mcu422", "gray", "base444")


@pytest.mark.gpu
@pytest.mark.skipif(not _have("example_b200"), reason="oracle/_ref not built")
def test_reference_example_decodes_through_the_helpers_on_the_cuda_back_end(jpegs, tmp_path):
    """example.c: jpeg_read_header -> jpegqs_start_decompress (q6, n3, progress callback) ->
    jpeg_read_scanlines -> jpegqs_finish_decompress -> BMP, with real libjpeg doing the IDCT /
    colour conversion after the re-armed decoder (quantsmooth.h:2861-2876).  Same pixels, same
    progress lines as the all-CPU build (example_cpu, stored); and the device renderer
    (jpegqs --ppm) gives them too."""
    exe = os.path.join(CSRC, "jpegqs")
    for name in EXAMPLE_FILES:
        check_input(name, jpegs[name])
        want = reference_output(f"example_cpu/{name}")
        b = str(tmp_path / "b200.bmp")
        r2 = subprocess.run([os.path.join(REFDIR, "example_b200"), jpegs[name], b], capture_output=True, text=True,
                            env=_b200_env())
        assert r2.returncode == 0, r2.stderr
        assert r2.stdout == want["stdout"], name                  # the progress callback sequence
        assert file_digest(b) == want["bmp"], name
        ppm = str(tmp_path / "dev.ppm")
        assert subprocess.run([exe, "-q", "6", "-i", "0", "--ppm", jpegs[name], ppm]).returncode == 0
        assert _rgb_digest(ppm) == want["rgb"], name


def reference_outputs(tmpdir):
    """The inputs' digests and what refcli_cpu and example_cpu write for the cases above."""
    jpegs = make_real_jpegs(tmpdir)
    out = {f"input/{name}": file_digest(p) for name, p in jpegs.items()}
    cases = REFCLI_CASES + [(name, a.split()) for a, names in B200_CLI_CASES.items() for name in names]
    for name, args in cases:
        a = os.path.join(tmpdir, "cpu.jpg")
        subprocess.run([os.path.join(REFDIR, "refcli_cpu"), "-i", "0"] + args + [jpegs[name], a], check=True, capture_output=True)
        out[f"refcli_cpu/{name} {' '.join(args)}"] = file_digest(a)
    for name in EXAMPLE_FILES:
        a = os.path.join(tmpdir, "cpu.bmp")
        r = subprocess.run([os.path.join(REFDIR, "example_cpu"), jpegs[name], a], check=True, capture_output=True, text=True)
        out[f"example_cpu/{name}"] = {"stdout": r.stdout, "bmp": file_digest(a), "rgb": _rgb_digest(a)}
    r = subprocess.run([os.sys.executable, os.path.join(ROOT, "tools", "codec_difftest.py"), "77", "30", "--record"],
                       cwd=tmpdir, check=True, capture_output=True, text=True)
    out["codec_difftest/77 30"] = json.loads(r.stdout.splitlines()[-1])
    return out
