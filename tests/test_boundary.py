"""CPU: the C-ABI library builds, loads and exports every symbol include/covins_b200.h declares; the
product package never touches oracle/; without a GPU the product fails loudly instead of falling back."""
import ctypes
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    syms = []
    for h in sorted(os.listdir(os.path.join(ROOT, "include"))):
        txt = open(os.path.join(ROOT, "include", h)).read()
        syms += re.findall(r"CVB_API\s+[\w\s\*]+?\b(cvb_\w+)\s*\(", txt)
    return sorted(set(syms))


def test_library_exports_every_declared_symbol():
    import covins_b200
    if not os.path.exists(covins_b200.LIB_PATH):
        covins_b200.build()
    lib = ctypes.CDLL(covins_b200.LIB_PATH)
    syms = _declared_symbols()
    assert len(syms) >= 15
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, missing
    assert lib.cvb_version() >= 100


def test_python_signatures_cover_the_header():
    from covins_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared_symbols()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "covins_b200")
    bad = []
    for dp, _, fs in os.walk(pkg):
        if os.sep + "build" in dp:
            continue
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h", ".c")) or f == "Makefile":
                txt = open(os.path.join(dp, f), errors="ignore").read()
                if re.search(r"(from|import)\s+oracle|oracle/|libcovins_oracle|/root/reference", txt):
                    # doc-strings may *mention* the rule; flag only code-like uses
                    for line in txt.splitlines():
                        if re.search(r"^\s*(from|import)\s+oracle|#include\s+\".*oracle|libcovins_oracle|/root/reference",
                                     line):
                            bad.append((f, line.strip()))
    assert not bad, bad


def test_no_cpu_fallback_without_gpu():
    # a child process with every device hidden, so that the check also runs where a GPU is present
    code = ("import covins_b200\n"
            "try:\n    covins_b200.Context(0)\nexcept covins_b200.CvbError:\n    raise SystemExit(0)\n"
            "raise SystemExit('a context was created without a CUDA device')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


def test_shard_rows_cuts_on_keyframe_boundaries():
    """host logic of the map-wide sharded k-NN (SURVEY §8e): contiguous, exhaustive, keyframe-aligned row ranges"""
    import numpy as np
    from covins_b200 import matching as M
    seg = np.array([0, 10, 10, 250, 600, 1000, 1001, 4000], np.int64)
    for world in (1, 2, 3, 8, 16):
        cuts = M.shard_rows(4000, world, seg)
        assert len(cuts) == world + 1 and cuts[0] == 0 and cuts[-1] == 4000
        assert np.all(np.diff(cuts) >= 0) and set(cuts.tolist()) <= set(seg.tolist())
    cuts = M.shard_rows(10, 4)                       # without keyframe boundaries: even split
    assert cuts.tolist() == [0, 2, 5, 7, 10]
