"""The C-ABI library loads and exports every symbol include/hns_b200.h declares (no compute calls: runs without a GPU)."""
import ctypes
import os
import re

import pytest

from hnanosolver_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "hns_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hns_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_functions():
    syms = declared_symbols()
    assert "hns_compute_sim" in syms and "hns_grid_create_from_coords" in syms and len(syms) >= 30


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_lib.LIB_PATH), "libhns_b200.so not built: python -m hnanosolver_b200.build"
    L = ctypes.CDLL(_lib.LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(L, s)]
    assert not missing, f"declared in include/hns_b200.h but not exported: {missing}"


def test_binding_table_matches_header():
    assert sorted(_lib.SIGNATURES) == declared_symbols()


def test_abi_version_and_error_channel():
    L = _lib.lib()
    assert L.hns_abi_version() == 1
    assert isinstance(L.hns_last_error(), bytes)


def test_no_cpu_fallback_when_library_missing(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libhns_b200.so")
    with pytest.raises(ImportError):
        _lib.lib()


def test_native_environment_switches():
    """The library reads only the switches whose two sides both stay in the product (each side is compared bit for bit by the tests)."""
    names = set()
    for dp, _, files in os.walk(os.path.join(ROOT, "hnanosolver_b200", "csrc")):
        for f in files:
            names |= set(re.findall(r"getenv\(\s*\"(HNS_[A-Z0-9_]+)\"", open(os.path.join(dp, f), errors="replace").read()))
    assert names == {"HNS_ADVECT4", "HNS_FUSED_COMBUSTION", "HNS_MG_GRAPH"}


def test_product_does_not_touch_the_oracle():
    pkg = os.path.join(ROOT, "hnanosolver_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dp, f), errors="replace").read()
                assert "liboracle" not in txt and "from oracle" not in txt and "import oracle" not in txt, os.path.join(dp, f)
