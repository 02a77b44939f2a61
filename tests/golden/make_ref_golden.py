"""Records tests/golden/ref_results.json.xz: what the UNMODIFIED reference objects (oracle/_ref, built by oracle/Makefile
from the reference's lib/*.cc where its sources exist) return for every input the tests give the `ref` fixture. Runs
those tests with AMB_TEST_RECORD_REF=1, which puts the live objects behind the fixture and merges each call's result
into the file. The gpu-marked one runs against the emulated library (tests/simt/library_emul.cc), as in
tests/test_emulated_gpu_suite.py. Nothing in the output is hand-edited.

    python tests/golden/make_ref_golden.py
"""
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
TESTS = ["tests/test_oracle_vs_ref.py", "tests/test_host_logic.py::test_geometry_matches_reference_blocks",
         "tests/test_library_simt.py::test_gr_adapter_split_blocks_preamble_then_slicer"]
GPU_TESTS = ["tests/test_gpu_parity.py::test_against_live_reference_if_present"]


def main():
    sys.path.insert(0, ROOT)
    from oracle import cpu_oracle
    if not cpu_oracle.ref_available():
        raise SystemExit("oracle/_ref/libairmodes_ref.so is not built: the reference sources are needed to record")
    out = os.path.join(HERE, "ref_results.json.xz")
    if os.path.exists(out):
        os.remove(out)
    env = dict(os.environ, AMB_TEST_RECORD_REF="1")
    pytest = [sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider"]
    subprocess.run(pytest + TESTS, env=env, cwd=ROOT, check=True)
    with tempfile.TemporaryDirectory() as tmp:
        lib = os.path.join(tmp, "libairmodes_b200_emulated.so")
        subprocess.run(["g++", "-std=c++17", "-O1", "-U_FORTIFY_SOURCE", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-Wno-psabi", "-shared", "-fPIC", "-o", lib,
                        os.path.join(ROOT, "tests", "simt", "library_emul.cc")], check=True)
        subprocess.run(pytest + ["-m", "gpu"] + GPU_TESTS, env=dict(env, AMB_TEST_EMULATED_LIB=lib), cwd=ROOT, check=True)
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
