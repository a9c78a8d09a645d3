"""CPU-side checks of the drop-in boundary: the shared library loads, exports every symbol
include/maxent_b200.h declares, and the ctypes mirrors of the structs have the C layout.
No compute calls (there is no GPU here)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "maxent_b200.h")


@pytest.fixture(scope="module")
def lib():
    from maxent_b200 import _lib, build
    build.build()
    return _lib.load()


def _declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"^\s*(?:const\s+)?[A-Za-z_][A-Za-z0-9_]*\s*\*?\s+\*?(mx_[a-z_A-Z0-9]+)\s*\(", src, flags=re.M)
    return sorted(set(names))


def test_header_functions_are_exported(lib):
    from maxent_b200 import _lib
    declared = _declared_functions()
    assert len(declared) >= 10
    bound = sorted(n for n, _, _ in _lib.SYMBOLS)
    assert declared == bound, "ctypes table and header disagree"
    for name in declared:
        assert hasattr(lib, name), name


def test_struct_layout_matches_c(tmp_path):
    """Compile a probe against the header with gcc and compare sizeof/offsetof with the ctypes mirrors."""
    from maxent_b200 import _lib
    structs = {"MxLMParams": _lib.MxLMParams, "MxProblem": _lib.MxProblem, "MxSweepOut": _lib.MxSweepOut}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "maxent_b200.h"', 'int main(void){']
    for sname, cls in structs.items():
        lines.append('printf("%s.sizeof %%zu\\n", sizeof(%s));' % (sname, sname))
        for fname, _ in cls._fields_:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (sname, fname, sname, fname))
    lines.append('printf("MX_MAX_NSV %d\\n", MX_MAX_NSV); printf("MX_N_ANALYZERS %d\\n", MX_N_ANALYZERS);')
    lines.append("return 0;}")
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    for sname, cls in structs.items():
        assert int(out[sname + ".sizeof"]) == ctypes.sizeof(cls)
        for fname, _ in cls._fields_:
            assert int(out["%s.%s" % (sname, fname)]) == getattr(cls, fname).offset, (sname, fname)
    assert int(out["MX_MAX_NSV"]) == _lib.MX_MAX_NSV
    assert int(out["MX_N_ANALYZERS"]) == _lib.N_ANALYZERS


def test_host_introspection_without_gpu(lib):
    """The two pure-host entry points work without a device; version string names the architecture."""
    assert b"sm_100a" in lib.mx_version()
    from maxent_b200 import _lib
    for s in (8, 32, 47, 52, 64):
        cfg = _lib.sweep_config(s)
        assert cfg["threads"] == 256
        assert 2 * (cfg["smem_bytes"] + 1024) <= 228 * 1024  # two 8-warp CTAs per SM
    sm = ctypes.c_int32()
    assert lib.mx_sweep_config(_lib.MX_MAX_NSV + 1, ctypes.byref(sm), None) == -2
    n = lib.mx_layout_V_size(1000, 52)
    assert n == 125 * 7 * 64
    assert lib.mx_layout_V_size(1000, 0) < 0


def test_product_has_no_cpu_fallback():
    """The product package never imports the oracle, and computing without a GPU raises."""
    pkg = os.path.join(ROOT, "maxent_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", txt, flags=re.M), f
    import torch
    if not torch.cuda.is_available():
        import numpy as np
        from maxent_b200 import engine, _lib
        with pytest.raises(_lib.MaxEntLibraryError):
            engine.SharedProblem(np.eye(4), 1.0, np.ones(4), np.ones(4))


def test_missing_library_is_loud(monkeypatch):
    from maxent_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libmaxent_b200.so")
    with pytest.raises(_lib.MaxEntLibraryError):
        _lib.load()


def test_torch_operators_registered_cuda_only():
    """The hot path is driven through torch.ops.maxent_b200.* (maxent_b200/ops.py): the three operators exist with
    caller-allocated outputs, and there is no CPU kernel behind them -- host tensors are refused by the dispatcher."""
    import torch
    from maxent_b200 import ops
    for name in ops.OPERATORS:
        schema = str(getattr(torch.ops.maxent_b200, name).default._schema)
        assert "(a!)" in schema and schema.endswith("-> ()"), schema
    t = torch.zeros((1, 4), dtype=torch.float64)
    with pytest.raises(NotImplementedError):
        ops.analyze(t[0], t, t, None, None, 0.2, 0, False, torch.zeros((1, 5), dtype=torch.int32), None, None)
    z = torch.zeros(4, dtype=torch.float64)
    with pytest.raises(NotImplementedError):
        ops.project_data(z, z, z, z, z, z, z, z, z, None, [2, 2, 2, 1, 0, 0, 0, 10, 0, 0, 0], [1.0, 1e-18, 1.3, 1e20, 1e-4, 1e-16, -1.0],
                         t, t, z)
