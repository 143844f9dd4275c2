"""Writes tests/golden/reference_outputs.json: what the UNMODIFIED reference gives for every case
the tests compare with it (file and coefficient outputs as SHA-256 digests), so that those tests
need no reference build.  Needs oracle/_ref, which oracle/Makefile builds from the reference's
sources, and the built product (the tests' inputs are written by its Pillow):

    python tests/golden/make_reference_outputs.py

Each test module computes its part in reference_outputs(); a key both compute must agree."""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import golden_io                  # noqa: E402
import oracle_lib as ol           # noqa: E402
import test_cli                   # noqa: E402
import test_gpu_edge              # noqa: E402
import test_oracle_vs_reference   # noqa: E402
import test_real_libjpeg          # noqa: E402


def main():
    ol.ensure_built()
    assert ol.have_ref("scalar"), "needs oracle/_ref (oracle/Makefile builds it from the reference's sources)"
    out = {}
    for mod in (test_oracle_vs_reference, test_gpu_edge, test_cli, test_real_libjpeg):
        with tempfile.TemporaryDirectory() as d:
            for k, v in mod.reference_outputs(d).items():
                assert out.setdefault(k, v) == v, k
    with open(golden_io.REFERENCE_OUTPUTS, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    print(len(out), "entries ->", golden_io.REFERENCE_OUTPUTS)


if __name__ == "__main__":
    main()
