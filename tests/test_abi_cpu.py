"""CPU: the C-ABI shared library builds, loads without a GPU driver, and exports every symbol include/b200parse.h
declares (no compute calls).  Plus the one host-only entry point (Pillow coefficient table) against the oracle."""
import ctypes
import re
from pathlib import Path

import numpy as np

from omniparser_b200 import _lib
from oracle import ref_restate as R

ROOT = Path(__file__).resolve().parents[1]


def _declared():
    text = (ROOT / "include" / "b200parse.h").read_text()
    return sorted(set(re.findall(r"\b(b2p_[a-z0-9_]+)\s*\(", text)))


def test_abi3_library_builds_and_exports_every_declared_symbol():
    _lib.build()
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    names = _declared()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/b200parse.h but not exported"
    assert set(_lib.PROTOTYPES) == set(names), set(_lib.PROTOTYPES) ^ set(names)
    assert _lib.lib().b2p_abi_version() == 3


def test_no_libcuda_link_dependency():
    """cudart is static and the driver API is resolved at run time, so the library loads on a GPU-less box."""
    import subprocess
    out = subprocess.run(["ldd", str(_lib.LIB_PATH)], capture_output=True, text=True).stdout
    assert "libcuda.so" not in out and "libcudart" not in out


def test_lanczos_coeff_table_equals_oracle():
    lib = _lib.lib()
    for (n_in, n_out) in [(1920, 640), (1080, 360), (3240, 640), (2160, 426), (300, 640), (200, 426), (1919, 640)]:
        ks = ctypes.c_int(0)
        cap = n_out * 64
        bounds = np.zeros((n_out, 2), np.int32)
        kk = np.zeros(cap, np.int32)
        rc = lib.b2p_lanczos_coeffs_host(n_in, n_out, ctypes.byref(ks), bounds.ctypes.data, kk.ctypes.data, cap)
        assert rc == 0
        rb, rk = R.lanczos_coeffs(n_in, n_out)
        assert ks.value == rk.shape[1]
        assert np.array_equal(bounds, rb)
        assert np.array_equal(kk[: n_out * ks.value].reshape(n_out, ks.value), rk)


def test_product_never_imports_oracle_or_standin():
    """The product path must not route through the oracle (or the seeded checkpoint definitions)."""
    import ast
    pkg = ROOT / "omniparser_b200"
    for f in pkg.glob("*.py"):
        tree = ast.parse(f.read_text())
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom) and node.module:
                names = [node.module]
            for n in names:
                assert not (n == "oracle" or n.startswith("oracle.") or n == "standin" or n.startswith("standin.")), (f.name, n)
