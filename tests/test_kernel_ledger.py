"""Every Chebyshev step-kernel instantiation built into ``libbdg.so`` has a case in ``variant_cases.LEDGER`` that
reaches it (``test_gpu_variants.py`` runs the cases), and the ledger names nothing the library lacks: an instantiation
added or removed fails here until it is assigned a case or taken out of the ledger."""

import os
import shutil
import subprocess

import pytest

from variant_cases import CASES, FAMILIES, LEDGER, short_names

LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bodge_b200", "libbdg.so")


def library_kernels():
    tool = shutil.which("cuobjdump") or ("/usr/local/cuda/bin/cuobjdump" if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)
    if not os.path.exists(LIB) or tool is None:
        pytest.skip("needs the built libbdg.so and cuobjdump")
    out = subprocess.run([tool, "-symbols", LIB], capture_output=True, text=True, check=True).stdout
    symbols = [line.split()[-1] for line in out.splitlines() if "STT_FUNC" in line and any(f in line for f in FAMILIES)]
    return short_names(symbols)


def test_the_ledger_is_exactly_the_library():
    found = library_kernels()
    assert len(found) == len(set(found)), "one short name for two kernels"
    missing = sorted(set(found) - set(LEDGER))
    stale = sorted(set(LEDGER) - set(found))
    assert not missing, f"{len(missing)} kernels in libbdg.so have no case: {missing}"
    assert not stale, f"{len(stale)} ledger entries are not in libbdg.so: {stale}"
    counts = {f: sum(k.startswith(f + "<") for k in found) for f in FAMILIES}
    assert counts == {"cheb_step_ell": 99, "cheb_step_dmma": 32, "cheb_step_fma": 8, "cheb_pair_step": 24, "cheb_cube_step": 6}


def test_every_ledger_case_exists():
    assert all(case in CASES for case in LEDGER.values())
    assert all(c.kernels for c in CASES.values())


def test_short_names_of_mangled_and_demangled_forms():
    mangled = "_ZN39_GLOBAL__N__626e5ff6_7_cheb_cu_93b4baa913cheb_step_fmaILi1ELb0EEEvPKiS2_PK7double2S5_PS3_iddPdPjS7_i"
    if shutil.which("c++filt") or shutil.which("cu++filt"):
        assert short_names([mangled]) == ["cheb_step_fma<1, false>"]
    plain = "void (anonymous namespace)::cheb_step_ell<8, 5, 1, true, false, false>(int const*, double*, RowWalk)"
    assert short_names([plain, "init_rademacher"]) == ["cheb_step_ell<8, 5, 1, true, false, false>"]
