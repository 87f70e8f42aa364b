"""The C-ABI library builds, loads, and exports every entry point declared in include/adapose_b200.h
(no compute calls here: this test runs without a GPU)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib_path():
    from rgbmanip_b200 import build
    return build.build()


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "adapose_b200.h")).read()
    return sorted(set(re.findall(r"ADP_API\s+[\w\s\*]+?\b(adp_\w+)\s*\(", src)))


def test_header_declares_entry_points():
    syms = declared_symbols()
    assert len(syms) >= 17 and "adp_conv_tc_run" in syms and "adp_fit" in syms


def test_library_exports_every_declared_symbol(lib_path):
    lib = ctypes.CDLL(lib_path)
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    assert not missing, missing
    lib.adp_abi_version.restype = ctypes.c_int
    from rgbmanip_b200 import _lib
    assert lib.adp_abi_version() == _lib.ADP_ABI_VERSION == int(re.search(r"#define ADP_ABI_VERSION (\d+)", open(os.path.join(ROOT, "include", "adapose_b200.h")).read()).group(1))


def test_binding_covers_the_header(lib_path):
    from rgbmanip_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared_symbols()
    _lib.load()


def test_sass_is_blackwell_native(lib_path):
    """tcgen05.mma -> UTCHMMA, TMA -> UTMALDG, tcgen05.ld -> LDTM in the shipped SASS (B200_PROFILING.md)."""
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    obj = os.path.join(ROOT, "rgbmanip_b200", "csrc", "build", "tc_conv.o")
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic
    assert "sm_100a" in subprocess.run([cuobjdump, "-lelf", lib_path], capture_output=True, text=True).stdout


def test_product_path_fails_loudly_without_cuda():
    """In a child process that sees no CUDA device, so that the check runs on GPU machines too."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, sys.argv[1])\n"
            "import pytest\n"
            "from rgbmanip_b200 import _lib, estimator\n"
            "with pytest.raises(_lib.AdpError):\n"
            "    estimator.AdaPoseEstimator_v5(None, {'load': False, 'direct_regression': True}, None)\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
