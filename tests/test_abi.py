"""CPU-side checks of the drop-in boundary: the C-ABI library builds for sm_100a, loads
without a GPU, exports every symbol include/comap_b200.h declares, and refuses to run
without a device (no CPU fallback)."""
import ctypes
import os
import re
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from comap_b200 import build, api
    build.build()
    return api.load()


def test_header_symbols_exported(lib):
    from comap_b200 import api
    hdr = open(os.path.join(ROOT, "include", "comap_b200.h")).read()
    declared = set(re.findall(r"\b(cmb_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(api.SYMBOLS)
    for s in declared:
        assert hasattr(lib, s), s


def test_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    h = ctypes.c_void_p()
    rc = lib.cmb_ctx_create(-1, None, ctypes.byref(h))
    assert rc != 0
    assert b"no CPU fallback" in lib.cmb_last_error()


def test_product_never_touches_oracle():
    """The product tree must not reference oracle/ (parity claims depend on it)."""
    pkg = os.path.join(ROOT, "comap_b200")
    for dp, _, fs in os.walk(pkg):
        if os.path.basename(dp) == "build":
            continue
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "liboracle" not in txt and "comap_oracle" not in txt and "oracle_binding" not in txt, f


# Environment switches the library may read: each forces a path production inputs also reach, or gives a test its
# reference (DESIGN.md s4, "Test switches").  A tuning choice is decided by measurement, not left to a switch.
TEST_SWITCHES = {"CMB_NULL_DEDUP", "CMB_NULL_DEDUP_HASH_BITS", "CMB_NULL_DEDUP_MIN_RUN", "CMB_K5_FILTER",
                 "CMB_K4_ALGO", "CMB_K1_PROTEIN", "CMB_DOWN_GLOBAL_TIPS"}


def test_library_reads_only_the_test_switches():
    csrc = os.path.join(ROOT, "comap_b200", "csrc")
    read = set()
    for f in os.listdir(csrc):
        read |= set(re.findall(r'getenv\("(CMB_\w+)"\)', open(os.path.join(csrc, f)).read()))
    assert read == TEST_SWITCHES
