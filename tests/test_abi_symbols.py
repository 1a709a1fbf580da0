"""CPU-side checks of the drop-in boundary: the shared library builds (nvcc cross-compiles
without a GPU), loads, and exports exactly the mrl_* symbols include/mrl_b200.h declares; argument errors are
reported through return codes + mrl_last_error (no exception crosses the ABI); and nothing under
modular_rl_b200/ imports the oracle.  No compute call is made here."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from modular_rl_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.lib()


def _declared():
    src = open(os.path.join(ROOT, "include", "mrl_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mrl_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported_and_bound(lib):
    from modular_rl_b200 import _lib
    names = _declared()
    assert len(names) >= 35
    for n in names:
        assert hasattr(lib, n), f"{n} declared in mrl_b200.h but not exported"
    assert set(names) == set(_lib.exported_symbols()), set(names) ^ set(_lib.exported_symbols())
    assert lib.mrl_version() >= 100


def test_library_exports_only_declared_symbols(lib):
    from modular_rl_b200 import _lib
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], check=True, capture_output=True, text=True).stdout
    exported = sorted({f[-1] for f in (line.split() for line in out.splitlines()) if f and f[-1].startswith("mrl_")})
    assert exported == _declared(), set(exported) ^ set(_declared())


def test_argument_errors_are_return_codes(lib):
    h = C.c_void_p()
    dims = (C.c_int * 3)(4, 300, 2)          # hidden width above the fused-kernel limit
    rc = lib.mrl_net_create(C.byref(h), 0, 2, dims, 1, 0)
    assert rc != 0 and b"width" in lib.mrl_last_error()
    dims = (C.c_int * 3)(4, 8, 2)
    assert lib.mrl_net_create(C.byref(h), 0, 2, dims, 2, 0) != 0     # value head needs dout 1
    assert b"value head" in lib.mrl_last_error()
    assert lib.mrl_net_create(C.byref(h), 0, 9, dims, 0, 0) != 0     # too many layers
    assert lib.mrl_batch_create(C.byref(h), 0, 0, 1) != 0
    assert lib.mrl_net_num_params(None) == -1


def test_product_code_never_imports_the_oracle():
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "modular_rl_b200")):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M):
                    bad.append(f)
    for f in ("run_pg.py",):
        p = os.path.join(ROOT, f)
        if os.path.exists(p) and re.search(r"^\s*(from|import)\s+oracle\b", open(p).read(), flags=re.M):
            bad.append(f)
    assert not bad, bad


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from modular_rl_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.lib()
