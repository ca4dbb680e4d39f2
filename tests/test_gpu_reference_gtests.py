"""The reference's OWN googletest suites (dietgpu/ans/ANSTest.cu:243-282, dietgpu/float/FloatTest.cu:
270-311), compiled unchanged against libdietgpu_b200.so through the include-path shim tests/ref_shim ->
include/dietgpu_b200_compat.hpp.  SURVEY.md section 8f-1's acceptance line: ANSTest and FloatTest pass
against the new library.

Their sources belong to the reference and are not part of this repository: `oracle/build_ref.sh gtests`,
run by __graft_entry__.build() where the reference's sources are present, compiles them into oracle/_ref/,
and a missing binary is a failure here.  The same cases, written for this repository, also run through
tests/test_gpu_compat.py."""
import os
import subprocess

import pytest

REF_BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref")


def _run(name, expect_tests):
    exe = os.path.join(REF_BIN, name)
    if not os.path.exists(exe):
        pytest.fail(f"{exe} missing: `oracle/build_ref.sh gtests` builds it where the reference's sources are present")
    p = subprocess.run([exe, "--gtest_color=no"], capture_output=True, text=True, timeout=900)
    out = p.stdout + p.stderr
    assert p.returncode == 0, out[-4000:]
    assert "[  PASSED  ]" in out and "FAILED" not in out, out[-4000:]
    for t in expect_tests:
        assert f"[       OK ] {t}" in out, (t, out[-4000:])


@pytest.mark.gpu
def test_reference_ans_gtest_unchanged():
    _run("ref_ans_test", ["ANSTest.ZeroSized", "ANSTest.BatchPointer", "ANSTest.BatchPointerLarge", "ANSTest.BatchStride"])


@pytest.mark.gpu
def test_reference_float_gtest_unchanged():
    _run("ref_float_test", ["FloatTest.Batch", "FloatTest.LargeBatch", "FloatTest.BatchSize1"])
