"""CPU checks of the drop-in boundary: the C-ABI library loads, exports every symbol include/mpp.h
declares, and fails loudly (no fallback) when there is no B200."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


def header_functions():
    src = open(os.path.join(ROOT, "include", "mpp.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mpp_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from maaco_path_planing_b200 import _lib
    L = ctypes.CDLL(_lib.SO_PATH)
    names = header_functions()
    assert len(names) >= 10
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, f"declared in mpp.h but not exported: {missing}"
    undeclared = [n for n in _lib.declared_symbols() if n not in names]
    assert not undeclared, f"bound in _lib.py but not declared in mpp.h: {undeclared}"
    unbound = [n for n in names if n not in _lib.declared_symbols()]
    assert not unbound, f"declared in mpp.h but not bound in _lib.py: {unbound}"


def header_prototypes():
    """name -> number of parameters, parsed from include/mpp.h."""
    src = open(os.path.join(ROOT, "include", "mpp.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for m in re.finditer(r"\b(mpp_[a-z0-9_]+)\s*\(([^;{}]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args in ("", "void") else args.count(",") + 1
    return out


def test_ctypes_signatures_match_header_arity():
    """Every binding in _lib.py passes exactly as many arguments as the prototype in mpp.h takes (a stale
    binding would shift every later argument and still load)."""
    from maaco_path_planing_b200 import _lib
    protos = header_prototypes()
    bad = {n: (len(sig[1]), protos.get(n)) for n, sig in _lib._SIGS.items() if protos.get(n) != len(sig[1])}
    assert not bad, f"(ctypes argtypes, header parameters) differ: {bad}"


def test_abi_version_3_and_error_string():
    from maaco_path_planing_b200 import _lib
    L = _lib.lib()
    assert L.mpp_abi_version() == 3
    assert isinstance(L.mpp_last_error(), bytes)


def test_q0_schedule_matches_oracle():
    import pyoracle as O
    from maaco_path_planing_b200 import _lib
    L = _lib.lib()
    for K in (1, 7, 10, 100, 333):
        for k in range(1, K + 1):
            for q in (0.5, 0.9, 0.05):
                assert L.mpp_maaco_q0(K, k, q) == O.lib().orc_maaco_q0(K, k, q)


def test_no_cpu_fallback():
    """Without a B200 the product must raise, not compute on the CPU."""
    import torch
    from maaco_path_planing_b200 import _lib, GridMap
    if torch.cuda.is_available() and _lib.lib().mpp_device_count() > 0:
        pytest.skip("a B200 is present")
    import numpy as np
    g = np.zeros((4, 4), int)
    g[0, 0], g[3, 3] = 2, 3
    with pytest.raises(_lib.MppError):
        GridMap(g, device=0)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "maaco_path_planing_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "pyoracle" not in txt and "mpp_oracle" not in txt and "ref_harness" not in txt, f
