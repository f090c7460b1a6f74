"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol
include/b200_search.h declares; the product never touches oracle/; compute calls fail loudly
without a GPU (no CPU fallback)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gpu_visible():
    """Whether CUDA sees a device in this process.  Asks CUDA (through torch, independent of the library under test):
    device nodes are not always numbered from /dev/nvidia0, and CUDA_VISIBLE_DEVICES can hide a device that exists."""
    import torch
    return torch.cuda.device_count() > 0


def test_library_exports_every_declared_symbol():
    from myscaledb_b200 import _lib
    L = _lib.lib()
    syms = _lib.declared_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/b200_search.h but not exported"
    assert b"sm_100a" in L.b200_version()


def test_product_never_references_oracle():
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "myscaledb_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".hpp")) or f == "Makefile":
                text = open(os.path.join(dirpath, f), errors="replace").read()
                if re.search(r"\boracle\b", text) and "no Python / CPU implementation" not in text:
                    for ln in text.split("\n"):
                        if re.search(r"(import|include|from|dlopen|CDLL).*oracle", ln):
                            bad.append((f, ln))
    assert not bad, bad


def test_sass_is_blackwell_native():
    so = os.path.join(ROOT, "myscaledb_b200", "libb200search.so")
    out = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    assert "sm_100a" in out or "SM100a" in out.upper() or "EF_CUDA_SM100" in out
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in out, f"{mnemonic} missing from SASS: the tcgen05/TMA path did not compile"


@pytest.mark.skipif(_gpu_visible(), reason="only meaningful without a GPU")
def test_compute_fails_loudly_without_gpu():
    import myscaledb_b200 as b2
    with pytest.raises(b2.B200Error) as ei:
        b2.flat_knn(b2.L2, np.zeros((1, 4), np.float32), np.zeros((4, 4), np.float32), 2)
    assert ei.value.code == 4 and "no CPU fallback" in str(ei.value)
    with pytest.raises(b2.B200Error):
        b2.Corpus(b2.IP, 64)


def test_reference_call_sites_compile_against_the_shim():
    """tests/cpp/callsite_compile.cpp pastes the call expressions of VIWithDataPart.cpp / BruteForceSearch.h /
    TantivyIndexStore.cpp; it must compile with -Werror against shim/b200_search_shim.hpp and link against the C ABI."""
    exe = os.path.join(ROOT, "tests", "cpp", "callsite_compile")
    subprocess.check_call(["g++", "-std=c++20", "-O1", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "shim"), os.path.join(ROOT, "tests", "cpp", "callsite_compile.cpp"), "-o", exe,
                           "-L" + os.path.join(ROOT, "myscaledb_b200"), "-lb200search",
                           "-Wl,-rpath,$ORIGIN/../../myscaledb_b200"])
    assert os.path.exists(exe)
    if not _gpu_visible():
        r = subprocess.run([exe], capture_output=True, text=True)
        assert r.returncode == 2 and "no CPU fallback" in r.stdout  # loud failure through SearchIndexException
