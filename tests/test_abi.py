"""The C-ABI library loads and exports every symbol include/kgpu.h declares
(no compute calls: this runs without a GPU)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

from kubegpu_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "kgpu.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(kgpu_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def built_lib():
    if not os.path.exists(_lib.LIB_PATH):
        subprocess.check_call(["make", "-s", "-C", ROOT, "kubegpu_b200/lib/libkgpu.so"])
    return ctypes.CDLL(_lib.LIB_PATH)


def test_header_and_binding_agree():
    assert header_symbols() == sorted(_lib.SYMBOLS)


def test_library_exports_every_declared_symbol(built_lib):
    for name in header_symbols():
        assert hasattr(built_lib, name), name


def test_version_and_error_path_without_device(built_lib):
    L = _lib.load()
    assert L.kgpu_version().decode() == "0.2.0"
    # bad arguments are rejected before any CUDA call
    h = ctypes.c_void_p()
    assert L.kgpu_create(None, 0, ctypes.byref(h)) == _lib.ERR_INVALID
    assert b"device ids" in L.kgpu_last_error(None)
    assert L.kgpu_create((ctypes.c_int * 1)(0), 1, None) == _lib.ERR_INVALID
    assert L.kgpu_set_variant(None, 2) == _lib.ERR_INVALID
    assert L.kgpu_num_nodes(None) == 0 and L.kgpu_destroy(None) == _lib.OK


def test_no_cpu_fallback_without_cuda(built_lib):
    """Product rule: without a CUDA device creating a scorer fails loudly.  A fresh process with every device
    hidden, so the rule is checked on a machine with a GPU too."""
    code = ("from kubegpu_b200.scorer import KgpuError, Scorer\n"
            "try:\n    Scorer()\nexcept KgpuError as e:\n    print(e.code, e)\n")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.startswith("%d " % _lib.ERR_CUDA) and "no CPU path" in out.stdout, out.stdout


def test_product_does_not_touch_oracle():
    """Nothing under kubegpu_b200/ may reference oracle/ (grading rule)."""
    pkg = os.path.join(ROOT, "kubegpu_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".cc", ".h", ".cpp")):
                text = open(os.path.join(dirpath, fn), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), fn
                assert "oracle_b" not in text and "oracle_a" not in text and "oracle/" not in text, fn


def test_few_pod_kernel_stages_tiles_with_tma():
    """The few-pod instantiations of the headline kernel (score_pairs_sparse<..., STREAM, TMA = 7 | 8>) must carry the
    bulk-copy and mbarrier instructions in their SASS (UBLKCP / SYNCS: B200_PROFILING.md's mnemonics for cp.async.bulk
    and mbarrier): the TMA path is compiled in, not a fallback to plain loads."""
    import shutil
    import subprocess
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    fn, counts = None, {}
    for line in sass.splitlines():
        if "Function :" in line:
            fn = line.split("Function :")[1].strip()
        elif fn and ("UBLKCP" in line or "SYNCS.PHASECHK" in line):
            counts[fn] = counts.get(fn, 0) + 1
    tma = [f for f in counts if "score_pairs_sparse" in f and ("ELi7E" in f or "ELi8E" in f)]
    assert len(tma) == 4, sorted(counts)          # byte / general keys x 7 / 8 blocks per SM
    assert all(counts[f] >= 4 for f in tma)       # three bulk copies per slab + the phase wait, at least
