"""CPU-only checks of the drop-in boundary: the C-ABI library loads without a GPU, exports every symbol that
include/fdjac_b200.h declares (and nothing is silently missing from the ctypes table), host-side scalar helpers agree
with the oracle, and compute entry points FAIL LOUDLY without a device (no CPU fallback)."""
import ctypes as C
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _build_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("_fdjac_build", ROOT / "finitediff.jl_b200" / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    _build_module().build()
    import _bootstrap
    return _bootstrap.load_package()


def _declared(header: str):
    text = (ROOT / "include" / header).read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(fdbs?_[a-z0-9_]+)\s*\(", text)))


def _exported(lib: Path):
    out = subprocess.run(["nm", "-D", "--defined-only", str(lib)], capture_output=True, text=True, check=True).stdout
    return {ln.split()[-1] for ln in out.splitlines() if " T " in ln}


def test_header_symbols_exported_and_bound(pkg):
    L = pkg._lib
    declared = _declared("fdjac_b200.h")
    assert len(declared) >= 25
    exported = _exported(L.LIB_PATH)
    missing = [s for s in declared if s not in exported]
    assert not missing, f"declared in include/fdjac_b200.h but not exported: {missing}"
    assert sorted(L.ABI_SYMBOLS) == declared, "ctypes table and header disagree"
    lib = L.lib()                      # binds every symbol; AttributeError if one is absent
    assert lib.fdb_abi_version() == 2


def test_synth_header_symbols(pkg):
    L = pkg._lib
    declared = [s for s in _declared("fdjac_synth.h") if not s.endswith("_ctx")]
    exported = _exported(L.SYNTH_PATH)
    assert not [s for s in declared if s not in exported]
    assert sorted(L.SYNTH_SYMBOLS) == sorted(declared)
    L.synth()


def test_sm100a_only(pkg):
    # the toolkit that built the library, found the way build.py finds nvcc (PATH need not contain the CUDA bin directory)
    cuobjdump = shutil.which("cuobjdump") or str(Path(_build_module().nvcc_path()).with_name("cuobjdump"))
    out = subprocess.run([cuobjdump, "--list-elf", str(pkg._lib.LIB_PATH)], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_step_size_helpers_match_oracle(pkg, oracle):
    lib = pkg._lib.lib()
    for fd in (0, 1):
        assert lib.fdb_default_relstep(fd) == oracle.default_relstep(fd)
        for xv in (-4.0, 0.0, 1e-30, 3.5e10):
            for d in (1.0, -1.0):
                assert lib.fdb_compute_epsilon(fd, xv, 1e-3, 1e-8, d) == oracle.compute_epsilon(fd, xv, 1e-3, 1e-8, d)
    assert pkg.default_relstep("forward") == 1.4901161193847656e-08      # sqrt(eps)
    assert pkg.default_relstep("central") == 6.0554544523933395e-06      # cbrt(eps)
    with pytest.raises(ValueError):
        pkg.default_relstep("hcentral2")


def test_no_cpu_fallback(pkg):
    """Without a GPU every compute entry point must fail with FDB_ERR_NO_DEVICE — never route to a CPU path."""
    L = pkg._lib
    if L.lib().fdb_device_count() > 0:
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    o = L.PlanOpts()
    cp = np.array([1, 2, 3], dtype=np.int64)
    rv = np.array([1, 2], dtype=np.int64)
    st = L.lib().fdb_plan_create_csc(C.byref(h), 2, 2, cp.ctypes.data, rv.ctypes.data, 0, None, None, 0, None, C.byref(o))
    assert st == L.FDB_ERR_NO_DEVICE and h.value is None
    assert b"no CPU fallback" in L.lib().fdb_last_error()
    assert L.lib().fdb_plan_create_dense(C.byref(h), 2, 2, 2, C.byref(o)) == L.FDB_ERR_NO_DEVICE
    assert L.lib().fdb_plan_create_banded(C.byref(h), 2, 2, 1, 1, 2, 0, None, C.byref(o)) == L.FDB_ERR_NO_DEVICE
    import torch
    with pytest.raises(TypeError):
        pkg.JacobianCache(torch.zeros(3, dtype=torch.float64), "forward")


def test_product_never_imports_oracle():
    """The product package must not reference oracle/ (only tests/, smoke() and bench.py may)."""
    for p in (ROOT / "finitediff.jl_b200").rglob("*"):
        if p.suffix in (".py", ".cu", ".cuh", ".h", ".jl"):
            txt = p.read_text()
            assert "fd_oracle" not in txt and "libfd_oracle" not in txt, p
            assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), p


def test_every_environment_switch_is_documented():
    """The A/B switches are read with getenv when a plan is created; DESIGN.md §4 is the only place a user can learn about
    them — a switch added to the sources must appear in that table."""
    import re
    root = Path(__file__).resolve().parent.parent
    names = set()
    for src in sorted((root / "finitediff.jl_b200" / "csrc").glob("*.cu*")):
        names |= set(re.findall(r'(?:getenv|env_is)\("(FDB[A-Z_0-9]*)"', src.read_text()))
    assert names, "no switches found: the scan is broken"
    design = (root / "DESIGN.md").read_text()
    missing = sorted(n for n in names if n not in design)
    assert not missing, f"undocumented environment switches: {missing}"
