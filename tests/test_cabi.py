"""CPU: the C-ABI library loads and exports every symbol include/b200rec.h declares; the Python binding table
matches the header; product code never imports the oracle; without a CUDA device calls fail loudly."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200rec.h")


def header_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b200_[A-Za-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from recsys2019_deeplearning_evaluation_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    syms = header_symbols()
    assert len(syms) >= 10
    for s in syms:
        assert hasattr(lib, s), "libb200rec.so does not export %s" % s


def test_binding_table_matches_header():
    from recsys2019_deeplearning_evaluation_b200 import _lib
    assert sorted(_lib.SIGNATURES) == header_symbols()
    lib = _lib.load()
    assert lib.b200_version() >= 100
    assert lib.b200_launch_count() >= 0


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "recsys2019_deeplearning_evaluation_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "ref_loader" not in txt, f


_WITHOUT_CUDA = """
from recsys2019_deeplearning_evaluation_b200 import _lib
from recsys2019_deeplearning_evaluation_b200.similarity import Compute_Similarity_Cython
from recsys2019_deeplearning_evaluation_b200.synth import synth_urm
try:
    Compute_Similarity_Cython(synth_urm(50, 20, 0.2), topK=5)
except (_lib.B200Error, MemoryError) as ex:
    print("raised", type(ex).__name__)
"""


def test_fails_loudly_without_cuda():
    """In a process that sees no CUDA device (CUDA_VISIBLE_DEVICES empty), so that it also runs on a machine with one."""
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _WITHOUT_CUDA]
    r = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode == 0 and "raised" in r.stdout, r.stdout[-2000:]


def test_argument_errors_mirror_the_reference():
    from recsys2019_deeplearning_evaluation_b200.similarity import Compute_Similarity_Cython, Compute_Similarity
    from recsys2019_deeplearning_evaluation_b200.synth import synth_urm
    X = synth_urm(50, 20, 0.2)
    with pytest.raises(ValueError, match="not recognized"):
        Compute_Similarity_Cython(X, similarity="cosin")  # pyx:141-144
    with pytest.raises(ValueError, match="different number of rows"):
        Compute_Similarity_Cython(X, row_weights=np.ones(49))  # pyx:188-190
    with pytest.raises(ValueError):
        Compute_Similarity(X, use_implementation="fortran")  # Compute_Similarity.py:121
    Xbad = X.copy(); Xbad.data[0] = np.inf
    with pytest.raises(AssertionError):
        Compute_Similarity(Xbad)  # Compute_Similarity.py:44
