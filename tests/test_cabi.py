"""CPU tests (no GPU): the C-ABI library builds, loads and exports every symbol include/b200sql.h
declares; with no device the product fails loudly instead of falling back."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(b2):
    decl = b2.parse_header()
    assert len(decl) >= 60
    lib = ctypes.CDLL(b2.LIB_PATH)
    missing = [n for n in decl if not hasattr(lib, n)]
    assert missing == []
    assert b"sm_100a" in b2.lib.b2_version()


def test_header_cites_reference_for_every_section():
    src = open(os.path.join(ROOT, "include", "b200sql.h")).read()
    for tag in ("a1", "a2", "a3/a4/a5", "a6/a7", "a8", "a9", "a10", "a11", "a12", "(e)"):
        assert tag in src
    assert len(re.findall(r"\.scala:\d+", src)) >= 25


def test_built_for_sm_100a(b2):
    import subprocess
    from spark_rapids_b200 import build
    cuobjdump = os.path.join(os.path.dirname(build.NVCC), "cuobjdump")   # the toolkit that built the library; PATH may lack it
    out = subprocess.run([cuobjdump, "-lelf", b2.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_gpu_fails_loudly(b2):
    from tests.conftest import HAS_GPU
    if HAS_GPU:
        pytest.skip("a GPU is present")
    import numpy as np
    with pytest.raises(b2.B2Error) as ei:
        b2.Column.from_numpy(np.arange(4, dtype=np.int64))
    assert "no CPU fallback" in str(ei.value)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "spark-rapids_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "import oracle" not in text and "from oracle" not in text, f


def test_jni_shim_compiles_and_binds_only_declared_entry_points():
    """jni/b2_jni.c is real source: it must pass a syntax check (against the stub jni.h when no JDK is present) and every
    b2_* function it calls must be declared in include/b200sql.h"""
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run(["make", "-C", os.path.join(root, "jni"), "check"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    src = open(os.path.join(root, "jni", "b2_jni.c")).read()
    called = set(re.findall(r"\b(b2_[a-z0-9_]+)\s*\(", src)) - {"b2_throw"}
    from spark_rapids_b200 import parse_header
    declared = set(parse_header())
    assert called <= declared, sorted(called - declared)
    natives = re.findall(r"JNICALL\s+(Java_[A-Za-z0-9_]+)", src)
    assert len(natives) >= 18 and len(set(natives)) == len(natives)
