"""CPU-only checks of the drop-in boundary: the C-ABI library builds, loads, and exports exactly the
symbols include/satb200.h declares; the product package never touches the oracle and fails loudly
without a GPU."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "satb200.h")
PKG = os.path.join(ROOT, "ppo-rl-satellite_b200")


def declared_symbols():
    src = open(HEADER, encoding="utf-8").read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sat_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib_path():
    import importlib.util
    spec = importlib.util.spec_from_file_location("satb200_build", os.path.join(PKG, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def test_header_symbols_are_exported(lib_path):
    out = subprocess.run(["nm", "-D", "--defined-only", lib_path], capture_output=True, text=True, check=True).stdout
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    decl = declared_symbols()
    assert len(decl) >= 20
    missing = [s for s in decl if s not in exported]
    assert not missing, f"declared in satb200.h but not exported: {missing}"
    extra = sorted(s for s in exported if s.startswith("sat_") and s not in decl)
    assert not extra, f"exported but not declared: {extra}"


def header_abi_version():
    m = re.search(r"^#define\s+SATB200_ABI_VERSION\s+(\d+)\s*$", open(HEADER, encoding="utf-8").read(), flags=re.M)
    assert m, "SATB200_ABI_VERSION not found in satb200.h"
    return int(m.group(1))


def test_ctypes_binding_covers_header_and_matches_header_abi_version(lib_path):
    """the binding declares every header symbol, and the header, the library and the binding agree on the ABI version
    (the version changes with any signature change, e.g. 3: sat_gae / sat_gae_flat take double gamma, lamda)"""
    from ppo_rl_satellite_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared_symbols()
    lib = _lib.load()                      # dlopen + symbol lookup, no compute
    assert lib.sat_abi_version() == header_abi_version() == _lib.ABI_VERSION >= 3
    assert lib.sat_strerror(0) == b"ok" and b"NULL" in lib.sat_strerror(-1)
    assert lib.sat_workspace_bytes(65536) >= 65536 // 32 * 19 * 16
    p = _lib.default_params()
    assert (p.d_range, p.u_grav, p.r_cw[0], p.v_cw[1], p.reset_p[0], p.reset_e[0]) == \
           (100000.0, 3.986e14, 27098000.0, 1970.0, 200000.0, 18000.0)


def test_struct_layouts_match_header(lib_path, tmp_path):
    """sizeof/offsetof of the POD structs as the C compiler sees them vs the ctypes mirrors."""
    import ctypes as C
    from ppo_rl_satellite_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "satb200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(SatEnvState),sizeof(SatEnvParams),sizeof(SatActorWeights),offsetof(SatEnvParams,stm),'
                   'offsetof(SatEnvParams,reset_e),offsetof(SatActorWeights,max_action));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(t) for t in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(_lib.SatEnvState), C.sizeof(_lib.SatEnvParams), C.sizeof(_lib.SatActorWeights),
            _lib.SatEnvParams.stm.offset, _lib.SatEnvParams.reset_e.offset, _lib.SatActorWeights.max_action.offset]
    assert got == want


def test_product_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from ppo_rl_satellite_b200 import engine, _lib
    with pytest.raises(_lib.SatError, match="no CPU fallback"):
        engine.EnvBatch(4)
    with pytest.raises(_lib.SatError):
        engine.rk4_propagate(torch.zeros((6, 4), dtype=torch.float64), 1.0, 1)


def test_product_never_imports_the_oracle():
    """the oracle is test infrastructure: nothing under the package (or the alias) may reference it."""
    bad = []
    for base in (PKG, os.path.join(ROOT, "ppo_rl_satellite_b200")):
        for dp, _dn, fns in os.walk(base):
            for fn in fns:
                if fn.endswith((".py", ".cu", ".cuh", ".h")):
                    txt = open(os.path.join(dp, fn), encoding="utf-8").read()
                    if re.search(r"^\s*(from|import)\s+oracle\b|sat_oracle|libsat_oracle|/root/reference", txt, flags=re.M):
                        bad.append(os.path.join(dp, fn))
    assert not bad, bad
