"""The C-ABI shared library loads without a GPU and exports every symbol that
include/oxli_b200.h declares; the ctypes table matches the header."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols() -> list[str]:
    text = open(os.path.join(ROOT, "include", "oxli_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(oxg_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_something():
    syms = declared_symbols()
    assert len(syms) >= 30 and "oxg_consume_batch" in syms


def test_library_exports_every_declared_symbol():
    from oxli_b200 import _build

    lib = ctypes.CDLL(_build.build_cuda())
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    assert not missing, missing


def test_ctypes_table_matches_header():
    from oxli_b200 import _capi

    assert sorted(_capi.SIGNATURES) == declared_symbols()


def test_no_cpu_fallback_without_gpu():
    from oxli_b200 import _capi

    if _capi.lib.oxg_device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(_capi.OxliCudaError):
        _capi.Table(21)
    assert _capi.lib.oxg_version() == b"0.3.0"


def test_product_never_imports_the_oracle():
    # the oracle is test infrastructure; the product tree must not reference it
    pkg = os.path.join(ROOT, "oxli_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "import oracle" not in text and "oxli_oracle" not in text, f


def test_specialised_k_list_is_sane():
    """csrc/klist.h drives both the build (one translation unit per k) and the dispatch in capi.cu."""
    from oxli_b200 import _build

    ks = _build.specialised_ks()
    assert ks == sorted(set(ks)) and all(1 <= k <= 64 for k in ks)
    assert {21, 31}.issubset(ks)  # the k values of BASELINE.json's configs; the only ones the route mode is built for
    text = open(os.path.join(_build.CSRC, "capi.cu")).read()
    assert "OXG_FOR_EACH_K(OXG_K_ENTRY)" in text and '#include "klist.h"' in text


def test_reference_suite_is_vendored_unmodified():
    """tests/reference_suite holds the reference's own tests byte for byte (their SHA-256 against
    tests/golden/reference_suite_sha256.json)."""
    import importlib.util
    import os

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_suite", "check_unmodified.py")
    spec = importlib.util.spec_from_file_location("check_unmodified", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert mod.main() == 0
