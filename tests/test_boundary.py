"""The drop-in boundary: the C-ABI library builds, loads and exports every symbol include/sie_b200.h declares;
the product never touches the oracle; struct layouts match the header.  No compute calls (no GPU here)."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "seaiceextentforecasting_b200")


def header_functions():
    src = open(os.path.join(ROOT, "include", "sie_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sie_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib_built):
    from seaiceextentforecasting_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = header_functions()
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/sie_b200.h but not exported"
    assert set(names) == set(_lib.EXPORTED_SYMBOLS)
    assert _lib.load().sie_abi_version() == _lib.ABI_VERSION == 2


def cuobjdump():
    """The cuobjdump of the toolkit whose nvcc builds the library (it need not be on PATH); the one on PATH where that
    nvcc is a wrapper outside the toolkit."""
    from seaiceextentforecasting_b200 import build
    beside = os.path.join(os.path.dirname(os.path.realpath(build._nvcc())), "cuobjdump")
    return beside if os.path.exists(beside) else shutil.which("cuobjdump") or beside


def test_library_is_sm100a_only(lib_built):
    from seaiceextentforecasting_b200 import _lib
    out = subprocess.run([cuobjdump(), "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_sass_has_dmma_and_bulk_copy(lib_built):
    from seaiceextentforecasting_b200 import _lib
    sass = subprocess.run([cuobjdump(), "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "DMMA.8x8x4" in sass          # FP64 tensor pipe in the correlation kernel
    assert "UBLKCP" in sass              # cp.async.bulk (TMA engine) operand staging
    assert "SYNCS" in sass               # mbarrier


def test_struct_layouts_match_header():
    from seaiceextentforecasting_b200 import _lib
    from seaiceextentforecasting_b200.forecast import GP_PROBLEM_DTYPE, GP_RESULT_DTYPE
    assert ctypes.sizeof(_lib.SieGpProblem) == 56 == GP_PROBLEM_DTYPE.itemsize
    assert ctypes.sizeof(_lib.SieGpResult) == 80 == GP_RESULT_DTYPE.itemsize
    for (name, _), f in zip(_lib.SieGpProblem._fields_, GP_PROBLEM_DTYPE.names):
        assert name == f and getattr(_lib.SieGpProblem, name).offset == GP_PROBLEM_DTYPE.fields[f][1]


def test_product_never_imports_oracle_or_reference():
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "/root/reference" not in txt, f


def test_product_raises_without_gpu_or_library():
    import torch
    from seaiceextentforecasting_b200 import _lib
    from seaiceextentforecasting_b200.ComplexNetworks import Network
    if torch.cuda.is_available():
        return
    n = Network(data=np.zeros((4, 4, 5)))
    try:
        Network.tau(n, 0.01)
    except _lib.SieError:
        pass
    else:
        raise AssertionError("no CPU fallback may exist")


def test_network_class_surface_matches_reference():
    """Constructor defaults / attribute names of ComplexNetworks.py:12-29, incl. the shared mutable defaults."""
    import inspect
    from seaiceextentforecasting_b200.ComplexNetworks import CN, Network
    sig = inspect.signature(Network.__init__)
    assert list(sig.parameters) == ["self", "data", "V", "A", "corrs", "tau", "nodes", "unavail", "anomaly", "links",
                                    "strength", "strengthmap"]
    n = Network(data=np.zeros((2, 3, 4)))
    assert (n.dimX, n.dimY, n.dimT) == (2, 3, 4)
    assert n.tau == 0 and callable(Network.tau) and callable(Network.area_level) and callable(Network.intra_links)
    assert list(inspect.signature(Network.tau).parameters) == ["self", "significance"]
    assert list(inspect.signature(Network.area_level).parameters) == ["self", "latlon_grid"]
    assert list(inspect.signature(Network.intra_links).parameters) == ["self", "area", "lat"]
    assert CN.Network is Network             # `from ComplexNetworks import CN` (north/June1st.py:197)


def test_reference_import_lines_resolve_through_compat():
    import importlib
    import sys
    compat = os.path.join(ROOT, "compat")
    sys.path.insert(0, compat)
    try:
        for m in ("ComplexNetworks", "CNs_backup", "CNs_backup.backups"):
            sys.modules.pop(m, None)
        CN = importlib.import_module("ComplexNetworks")             # import ComplexNetworks as CN
        from ComplexNetworks import CN as CN2                       # north/June1st.py:197
        from CNs_backup.backups import CN_forecast as CN3           # June1st_retro.py:198
        from seaiceextentforecasting_b200.ComplexNetworks import Network
        assert CN.Network is Network and CN2.Network is Network and CN3.Network is Network
    finally:
        sys.path.remove(compat)
        for m in ("ComplexNetworks", "CNs_backup", "CNs_backup.backups"):
            sys.modules.pop(m, None)
