"""CPU tests of the C-ABI boundary: the library builds, loads, and exports every declared symbol."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from dotaclient_b200 import _lib, build
    build.build()
    return _lib.load()


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "dotaclient_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dc_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported(lib):
    names = declared_symbols()
    assert len(names) >= 10
    for n in names:
        assert hasattr(lib, n), "declared in include/dotaclient_b200.h but not exported: " + n


def test_ctypes_signatures_cover_the_header():
    from dotaclient_b200 import _lib
    assert set(declared_symbols()) <= set(_lib.SIGNATURES)


def test_version_and_argument_errors_without_gpu(lib):
    assert lib.dc_version() >= 100
    # argument validation happens before any CUDA call, so it is testable on a CPU-only box
    rc = lib.dc_gae_scan(None, 0, None, None, 1, None, None, 0.98, 0.97, None, None, None)
    assert rc == -1 and b"dc_gae_scan" in lib.dc_last_error()
    rc = lib.dc_rnn_seq_fwd(7, None, None, None, None, None, 1, 1, 128, None, None)
    assert rc == -1 and b"unknown cell" in lib.dc_last_error()
    rc = lib.dc_rnn_seq_fwd(1, None, None, None, None, None, 1, 1, 130, None, None)
    assert rc == -2
    assert lib.dc_rnn_workspace_bytes(1, 7, 128) == 4 * 128 * 128 * 4
    assert lib.dc_rnn_workspace_bytes(0, 33, 256) == 2 * 2 * 8 * 32 * 256 * 4      # two clusters, ping-pong partials
    # the fused unit-encoder backward: null pointers / unsupported group sizes / misaligned operands are reported, nothing is launched
    one = 4096                                       # any non-null, 16-byte aligned "pointer": validation fails before it is used
    assert lib.dc_unit_wgrad_routed(None, None, 896, one, one, 8, 16, one, one, one, None) == -1 and b"dc_unit_wgrad_routed" in lib.dc_last_error()
    assert lib.dc_unit_wgrad_routed(one, None, 896, one, one, 8, 3, one, one, one, None) == -2          # 5 or 16 units only
    assert lib.dc_unit_wgrad_routed(one, None, 64, one, one, 8, 16, one, one, one, None) == -1          # row pitch below 128
    assert lib.dc_unit_dgrad_fused(one, None, 896, one, None, 40, None, None, one, one, one, 8, 16, one, one, 0, one, None) == -1   # no W^T
    assert lib.dc_unit_dgrad_fused(one, None, 896, one, None, 40, None, one, one, one, one, 8, 4, one, one, 0, one, None) == -2    # 1, 5 or 16
    assert lib.dc_unit_dgrad_fused(one, None, 896, None, None, 40, None, one, one, one, one, 8, 16, one, one, 0, one, None) == -1  # routing without arg-max
    assert lib.dc_unit_dgrad_fused(one, None, 896, one, one, 40, None, one, one, one, one, 8, 16, one, one, 0, one, None) == -1    # dlogits without att
    assert lib.dc_unit_dgrad_fused(one, None, 896, one, None, 40, None, one, one + 4, one, one, 8, 16, one, one, 0, one, None) == -1   # units misaligned
    assert b"dc_unit_dgrad_fused" in lib.dc_last_error()


def test_sass_is_sm100a_only():
    import subprocess
    from dotaclient_b200 import build
    so = os.path.join(ROOT, "dotaclient_b200", "libdotaclient_b200.so")
    cuobjdump = os.path.join(os.path.dirname(build._nvcc()), "cuobjdump")          # the toolkit that built the library
    out = subprocess.run([cuobjdump, "-lelf", so], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: no file of the product package may reference it."""
    pkg = os.path.join(ROOT, "dotaclient_b200")
    for base, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(base, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "reference_shim" not in text, f


def test_product_never_touches_the_oracle_or_the_reference():
    """oracle/ is test infrastructure: nothing under dotaclient_b200/ (nor the C sources) may import, load or mention it, and
    nothing shipped may read /root/reference at run time (it does not exist on the GPU box)."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "dotaclient_b200")
    offenders = []
    for d, _, files in os.walk(pkg):
        if os.path.basename(d) in ("build", "__pycache__"):
            continue
        for f in files:
            if not f.endswith((".py", ".cu", ".cuh", ".h")):
                continue
            text = open(os.path.join(d, f), encoding="utf-8", errors="replace").read()
            if re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M) or "oracle/" in text and f.endswith(".py") and "import" in text and \
                    re.search(r"(CDLL|open)\([^)]*oracle", text):
                offenders.append(os.path.join(d, f))
            if "/root/reference" in text:
                offenders.append(os.path.join(d, f) + " (reads /root/reference)")
    assert not offenders, offenders
    for name in ("bench.py", "__graft_entry__.py"):
        text = open(os.path.join(root, name), encoding="utf-8").read()
        assert "/root/reference" not in text, name
