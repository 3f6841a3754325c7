"""Runs the C++ restatement of the reference's unit tests (tests/cpp/test_reference_api.cc) — the host side
above the C ABI written in the reference's own language, through the reference-named interfaces."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "build", "test_reference_api")
BATCHER = os.path.join(ROOT, "tests", "cpp", "build", "test_stripe_batcher")


def test_cpp_binary_is_built():
    """CPU-side check: the binary exists (built by __graft_entry__.build()) and links against liblzgpu.so."""
    if not os.path.exists(BIN):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")], check=True)
    out = subprocess.run(["ldd", BIN], capture_output=True, text=True).stdout
    assert "liblzgpu.so" in out and "not found" not in out.split("liblzgpu.so")[1].split("\n")[0]


@pytest.mark.gpu
def test_reference_api_cpp():
    if not os.path.exists(BIN):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")], check=True)
    r = subprocess.run([BIN], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "passed" in r.stdout


def test_batcher_binary_is_built():
    if not os.path.exists(BATCHER):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")], check=True)
    out = subprocess.run(["ldd", BATCHER], capture_output=True, text=True).stdout
    assert "liblzgpu.so" in out and "liboracle.so" in out and "not found" not in out


@pytest.mark.gpu
def test_stripe_batcher_cpp():
    """lzgpu::StripeBatcher (include/lzgpu_stripe_batcher.hpp): the mount write path batched by stripe, checked block by
    block against the CPU oracle inside the C++ test (tests/cpp/test_stripe_batcher.cc)."""
    if not os.path.exists(BATCHER):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")], check=True)
    r = subprocess.run([BATCHER], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all tests passed" in r.stdout


READ_PLAN = os.path.join(ROOT, "tests", "cpp", "build", "test_read_plan")
READ_PLANS = os.path.join(ROOT, "tests", "golden", "read_plans.txt")


@pytest.mark.gpu
def test_read_plan_mirror_cpp():
    """lzgpu::SliceReadPlan (include/lzgpu_read_plan.hpp), the GPU-backed mirror of ReadPlan::postProcessData, on plans
    built by the reference's own ChunkReadPlanner (tests/golden/read_plans.txt) — must reproduce the reference's
    post-processed buffer byte for byte (tests/cpp/test_read_plan.cc)."""
    if not os.path.exists(READ_PLAN):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")], check=True)
    r = subprocess.run([READ_PLAN, READ_PLANS], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "16 plans, all tests passed" in r.stdout


def _run_cpu_build(name, *args):
    """The same C++ test source linked against tests/cpp/oracle_backend.cc (a test-only stand-in for the GPU entry points backed
    by the CPU oracle) instead of liblzgpu.so: covers the HOST logic of the header on a machine without a GPU."""
    exe = os.path.join(ROOT, "tests", "cpp", "build", name)
    if not os.path.exists(exe):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")], check=True)
    r = subprocess.run([exe, *args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all tests passed" in r.stdout


def test_stripe_batcher_host_logic_on_cpu():
    """slot bookkeeping, completeness, read-back blocks, write ids, packet prefixes of lzgpu::StripeBatcher"""
    _run_cpu_build("test_stripe_batcher_cpu")


def test_read_plan_mirror_host_logic_on_cpu():
    """part numbering, buffer layout, BlockConverter of lzgpu::SliceReadPlan on plans built by the reference's ChunkReadPlanner
    (tests/golden/read_plans.txt)"""
    _run_cpu_build("test_read_plan_cpu", READ_PLANS)


LINK_SUB = os.path.join(ROOT, "tests", "cpp", "build", "test_link_substitution")
LINK_SUB_CXX = os.path.join(ROOT, "tests", "cpp", "build", "test_link_substitution_cxx")


def _need_link_sub(exe):
    if not os.path.exists(exe):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")], check=False)
    if not os.path.exists(exe):
        pytest.skip("built only where /root/reference exists (the reference's unit-test sources are compiled in place)")


@pytest.mark.parametrize("exe", [LINK_SUB, LINK_SUB_CXX], ids=["isal_names", "cxx_names"])
def test_link_substitution_binaries_use_only_liblzgpu(exe):
    """The reference's own unit-test sources, linked: every GF / CRC / xor symbol must come from liblzgpu.so — no oracle, no
    reference objects for crc.cc / block_xor.cc / galois_field_*.cc in the link."""
    _need_link_sub(exe)
    ldd = subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    assert "liblzgpu.so" in ldd and "liblzref" not in ldd and "liboracle" not in ldd and "not found" not in ldd
    undefined = subprocess.run(["nm", "-C", "-u", exe], capture_output=True, text=True).stdout
    for name in ("ec_encode_data", "ec_init_tables", "gf_gen_rs_matrix", "gf_invert_matrix"):
        assert name in undefined, name  # resolved at load time by the shared library, not by an object of the reference
    if exe == LINK_SUB:
        for name in ("mycrc32(", "mycrc32_combine(", "blockXor("):
            assert name in undefined, name


@pytest.mark.gpu
@pytest.mark.parametrize("exe", [LINK_SUB, LINK_SUB_CXX], ids=["isal_names", "cxx_names"])
def test_reference_unit_tests_run_on_the_gpu_library(exe):
    """reed_solomon_unittest.cc, crc_unittest.cc, block_xor_unittest.cc, ec_read_plan_unittest.cc, xor_read_plan_unittest.cc of the
    reference (unmodified, compiled where they lie) with liblzgpu.so substituted at link time: all their expectations hold."""
    _need_link_sub(exe)
    r = subprocess.run([exe, "-Benchmark"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert "0 failed expectations" in r.stdout
    assert "ReedSolomon.TestRecovery" in r.stdout
    if exe == LINK_SUB:
        assert "ECReadPlanTests.VerifyRead1" in r.stdout and "CrcTests.MyCrc32" in r.stdout and "BlockXorTests.BlockXor" in r.stdout
