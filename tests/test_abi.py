"""The C-ABI library loads without a GPU and exports exactly what include/mmrs_b200.h declares."""
import ctypes
import re
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
HEADER = ROOT / "include" / "mmrs_b200.h"


def declared_symbols():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    return sorted(set(re.findall(r"\b(mmrs_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_something():
    syms = declared_symbols()
    assert "mmrs_search_topk" in syms and "mmrs_selfjoin_pairs" in syms and len(syms) >= 12


def test_library_exports_every_declared_symbol(mm):
    lib = ctypes.CDLL(str(mm._cabi.LIB_PATH))
    for s in declared_symbols():
        assert hasattr(lib, s), f"{s} declared in mmrs_b200.h but not exported"
    out = subprocess.run(["nm", "-D", "--defined-only", str(mm._cabi.LIB_PATH)], capture_output=True, text=True).stdout
    exported = sorted(l.split()[-1] for l in out.splitlines() if " T " in l and "mmrs_" in l)
    assert exported == declared_symbols(), "library exports symbols the header does not declare"


def test_python_binding_covers_the_header(mm):
    assert sorted(mm._cabi.SIGNATURES) == declared_symbols()


def test_abi_version_3_and_pure_host_queries(mm):
    lib = mm._cabi.lib
    assert lib.mmrs_abi_version() == mm._cabi.ABI_VERSION == 3
    # workspace queries are pure host arithmetic: usable without a device
    small = lib.mmrs_search_workspace_bytes(10_000, 512, 0, 100, 10)
    big = lib.mmrs_search_workspace_bytes(1_000_000, 512, 1, 256, 100)
    assert 0 < small < big
    assert lib.mmrs_search_host_staging_bytes(512, 16, 100) >= 16 * 512 * 4 + 16 * 100 * 12
    assert lib.mmrs_topk_merge_workspace_bytes(8, 256, 100) >= 8 * 256 * 100 * 8


def test_stale_library_is_refused(mm, tmp_path):
    """A library left over from ABI version 2 loads, but its entry points take other arguments: the
    loader must refuse it and name the rebuild."""
    src = tmp_path / "stale.cpp"
    src.write_text('extern "C" int mmrs_abi_version(void) { return 2; }\n')
    so = tmp_path / "libstale.so"
    subprocess.run(["g++", "-O1", "-shared", "-fPIC", str(src), "-o", str(so)], check=True)
    with pytest.raises(ImportError, match=r"version 2, this package needs 3.*build\.py --force"):
        mm._cabi.open_library(so)
    assert mm._cabi.open_library(mm._cabi.LIB_PATH).mmrs_abi_version() == 3


def test_no_cpu_fallback(mm):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU path"):
        mm.search_topk(torch.randn(2, 8), torch.randn(16, 8), 3)
    with pytest.raises(RuntimeError, match="no CPU path"):
        mm.find_duplicate_pairs(torch.randn(16, 8), 0.9)
    with pytest.raises(RuntimeError, match="no CPU path"):
        mm.get_similarity(torch.randn(16, 8), [0] * 16, 0, torch.randn(8))
    # the raw ABI refuses too (no device): status is an error code, never a silent result
    st = mm._cabi.lib.mmrs_device_check(0)
    assert st < 0 and mm._cabi.last_error()


def test_product_never_imports_the_oracle():
    pkg = ROOT / "multi-modal-retrieval-system-image-search-and-data-governance_b200"
    for f in pkg.glob("*.py"):
        text = f.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
        assert "oracle." not in text, f
