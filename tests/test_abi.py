"""CPU checks of the drop-in boundary: the C-ABI library loads, exports every symbol
include/conicip_b200.h declares, and the ctypes table mirrors the header.  No compute calls."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "conicip_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(cip_[a-z0-9_A-Z]+)\s*\(", src)))


def test_header_declares_the_protocol_levels():
    syms = declared_symbols()
    for s in ("cip_create", "cip_factor", "cip_solve", "cip_destroy", "cip_nt_scaling", "cip_maxstep",
              "cip_apply", "cip_cone_prod", "cip_cone_div", "cip_comm_init"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    import conicip_b200 as cb
    assert os.path.exists(cb.LIB_PATH), "build the library first (__graft_entry__.build())"
    L = ctypes.CDLL(cb.LIB_PATH)
    for s in declared_symbols():
        assert hasattr(L, s), f"{s} declared in the header but not exported"


def test_ctypes_table_matches_header():
    import conicip_b200 as cb
    assert sorted(cb.SIGNATURES) == declared_symbols()
    cb.lib()                                   # resolves and types every symbol
    assert cb.lib().cip_version() >= 100


def test_library_is_sm100a_native_with_tma_and_dmma():
    """SASS evidence that the hot kernel is the TMA-fed FP64 tensor-core path."""
    import conicip_b200 as cb
    # found where __graft_entry__.build() finds nvcc
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    try:
        sass = subprocess.run([cuobjdump, "-sass", "-fun", "gemm_nt_kernel", cb.LIB_PATH], capture_output=True,
                              text=True, timeout=120).stdout
    except FileNotFoundError:
        pytest.skip("cuobjdump not found")
    if "DMMA" not in sass:                      # -fun needs the mangled name on some versions
        sass = subprocess.run([cuobjdump, "-sass", cb.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    assert "sm_100a" in sass or "EF_CUDA_SM100" in sass
    assert "DMMA.8x8x4" in sass and "UTMALDG" in sass and "SYNCS" in sass


def test_no_oracle_import_in_product():
    """The product path must never route through the oracle (or any CPU fallback)."""
    pkg = os.path.join(ROOT, "conicip.jl_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "import oracle" not in src and "from oracle" not in src, fn


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    import conicip_b200 as cb
    from conicip_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(ImportError):
        _lib.lib()
