"""The C-ABI shared library builds for sm_100a, loads without a GPU and exports every symbol
include/seam_b200.h declares; compute entry points fail loudly when no device is present."""
import ctypes
import os
import subprocess

import pytest
import torch

import seam_match_rcnn_b200 as pkg


def test_library_builds_and_exports_all_declared_symbols():
    path = pkg.build_library()
    assert os.path.exists(path)
    lib = pkg.load_library()
    declared = pkg.declared_symbols()
    assert len(declared) >= 17
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} declared in include/seam_b200.h but not exported"
    assert lib.seam_abi_version() == 3
    from seam_match_rcnn_b200._lib import SeamExchange
    import ctypes
    assert ctypes.sizeof(SeamExchange) == lib.seam_exchange_sizeof(), "ctypes image of struct seam_exchange is out of step with the header"
    # pure host helpers are callable without a device
    assert lib.seam_aggregate_workspace_bytes(1000) >= 256       # the fused kernel needs no workspace
    assert lib.seam_nlb_workspace_bytes(3, 10) >= 2 * 30 * 256 * 4


def test_library_contains_blackwell_instructions():
    """SASS evidence that the hot kernels are tcgen05 / TMA code, not a recompiled legacy path."""
    cuobjdump = "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", pkg.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTMALDG", "UBLKCP", "LDTM"):
        assert mnemonic in sass, mnemonic


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    lib = pkg.load_library()
    h = ctypes.c_void_p()
    rc = lib.seam_create(ctypes.byref(h), 0)
    assert rc != 0 and not h.value
    assert b"no CUDA device" in lib.seam_last_error(None)
    with pytest.raises(pkg.SeamError):
        pkg.SeamEngine("cuda:0")
    with pytest.raises(pkg.SeamError):
        pkg.get_engine("cpu")
    m = pkg.TemporalAggregationNLB().eval()
    seq = torch.zeros(3, 2, 256)
    with pytest.raises(pkg.SeamError):
        m(None, None, None, x3_1_seq=seq, x3_1_mask=torch.zeros(2, 3, dtype=torch.bool), x3_2=torch.zeros(4, 256))
    with pytest.raises(pkg.SeamError):
        pkg.NONLocalBlock1D()(torch.zeros(1, 256, 4))


def test_product_package_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under seam-match-rcnn_b200/ may reference it."""
    root = os.path.dirname(pkg.LIB_PATH)
    for dirpath, _, files in os.walk(root):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "seam_oracle" not in text and "from oracle" not in text and "import oracle" not in text, f


def test_ctypes_bindings_match_the_header():
    """Every function declared in include/seam_b200.h is bound in _lib.py with as many arguments as the
    header gives it (a drifted binding would pass garbage through the C ABI without any error)."""
    import re
    header = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "seam_b200.h")
    with open(header) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    lib = pkg.load_library()
    seen = 0
    for m in re.finditer(r"\b(seam_[a-z_0-9]+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S):
        name, params = m.group(1), m.group(2).strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        fn = getattr(lib, name)
        assert fn.argtypes is not None, f"{name} has no argtypes in _lib.py"
        assert len(fn.argtypes) == n, f"{name}: header has {n} parameters, binding {len(fn.argtypes)}"
        seen += 1
    assert seen == len(pkg.declared_symbols())


def test_library_has_one_build_and_reads_no_environment():
    """The CUDA sources compile one way only: no preprocessor switch, no -D flag, and no environment variable
    that changes at run time what the library computes or how it partitions the work."""
    import re
    from seam_match_rcnn_b200 import _build
    assert not [f for f in _build.NVCC_FLAGS if f.startswith("-D")]
    for f in sorted(os.listdir(_build.CSRC)):
        if f.endswith((".cu", ".cuh")):
            with open(os.path.join(_build.CSRC, f)) as fh:
                text = fh.read()
            assert not re.search(r"^\s*#\s*(if|ifdef|ifndef)\b", text, flags=re.M), f"{f}: conditional compilation"
            assert "getenv" not in text, f"{f}: reads the environment"
