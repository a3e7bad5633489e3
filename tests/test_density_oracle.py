"""CPU checks behind ``Hamiltonian.density_matrix`` / ``order_parameter`` / ``selfconsistent``: the KPM reference
against the exact ``f(H)``, the sign of the gap equation against the reference's free energy, the Fermi series and its
length rule, and the new C-ABI entry points.  The GPU twin is ``test_gpu_density.py``."""

import os
import re

import numpy as np
import pytest

import fermi_oracle as fo
from bodge_b200 import _native, kpm, workloads
from oracle import bdg_oracle as orc
from util import oracle_assemble

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T = 0.1


def assembled(name, shape):
    _, (ptr, idx, dat) = oracle_assemble(shape, [getattr(workloads, name)(shape)])
    return orc.to_scipy(ptr, idx, dat), 1.01 * orc.norm_inf(ptr, idx, dat)


@pytest.mark.parametrize("name,shape", [("readme_swave", (6, 5, 1)), ("dwave_rashba", (5, 6, 1))])
def test_local_kpm_blocks_equal_dense_fermi(name, shape):
    H, scale = assembled(name, shape)
    rho = fo.fermi_dense(H.toarray(), T)
    Ly = shape[1]
    pairs = [(7, 7), (0, 0), (7, 8), (8, 7), (7, 7 + Ly), (13, 13 - Ly), (29, 28)]  # on-site and bonds
    j = np.array([p[1] for p in pairs])
    i = np.array([p[0] for p in pairs])
    uj, pos = np.unique(j, return_inverse=True)
    rows = (4 * uj[:, None] + np.arange(4)).ravel()
    read_col = (4 * pos[:, None] + np.arange(4)).ravel()
    n_coef = kpm.free_energy_moments(T, scale)[0]
    acc = fo.fermi_local_kpm(H, rows, read_col, np.repeat(i, 4), T, n_coef, scale)
    got = acc.reshape(len(pairs), 4, 4).transpose(0, 2, 1)
    want = np.stack([rho[4 * a:4 * a + 4, 4 * b:4 * b + 4] for a, b in pairs])
    assert np.max(np.abs(got - want)) <= 1e-10


def test_gap_equation_sign_is_hellmann_feynman():
    """∂F/∂Re Δ_k = 2 Re ρ[4k, 4k+3] and ∂F/∂Im Δ_k = 2 Im ρ[4k, 4k+3] for the reference's free energy, so the update
    Δ_i = -V ρ[4i, 4i+3] makes F + Σ|Δ_i|²/V stationary."""
    L, T_ = 4, 0.1
    rng = np.random.default_rng(5)
    delta = 0.2 * rng.random(L * L) * np.exp(2j * np.pi * rng.random(L * L))
    rho = fo.fermi_dense(fo.square_attractive(L, delta, mu=-0.7), T_)
    h = 1e-6
    for k in (0, 5, 10):
        for unit, part in ((1.0, np.real), (1j, np.imag)):
            dp, dm = delta.copy(), delta.copy()
            dp[k] += unit * h
            dm[k] -= unit * h
            fd = (orc.free_energy_dense(fo.square_attractive(L, dp, mu=-0.7), T_)
                  - orc.free_energy_dense(fo.square_attractive(L, dm, mu=-0.7), T_)) / (2 * h)
            assert abs(fd - 2 * part(rho[4 * k, 4 * k + 3])) <= 1e-7


def test_dense_gap_fixed_point():
    """The 6 x 6 open lattice (H[i,i] = σ0, bonds -σ0, V = 2, T = 0.05, start 0.1) has an edge-enhanced solution."""
    delta, it = fo.gap_fixed_point(6, 2.0, 0.05, tol=1e-10)
    assert 40 <= it <= 80
    assert 0.2 < np.min(np.abs(delta)) < np.max(np.abs(delta)) < 0.36
    assert abs(delta[0]) > abs(delta[2 * 6 + 2])  # corner above the centre


def test_fermi_coefficients_and_their_length():
    scale = 6.3
    for T_ in (0.05, 0.2, 1.0):
        n, reached = kpm.free_energy_moments(T_, scale, 1e-13)
        c = kpm.fermi_coefficients(T_, 2 * n, scale)
        assert reached == 1e-13
        assert np.max(np.abs(c[n:])) <= 1e-13  # what the length rule drops is below tol
        x = np.linspace(-1, 1, 101)
        series = np.polynomial.chebyshev.chebval(x, c[:n])
        assert np.max(np.abs(series - fo.fermi(scale * x, T_))) <= 1e-12
    assert np.allclose(kpm.fermi_coefficients(0.3, 64, 2.0), orc.cheb_coefficients(lambda e: fo.fermi(e, 0.3), 64, 2.0),
                       rtol=0, atol=1e-15)
    with pytest.raises(ValueError):
        kpm.fermi_coefficients(0.0, 64, 2.0)


def test_local_accumulator_symbols():
    header = open(os.path.join(REPO, "include", "bdg.h")).read()
    for name in ("bdg_cheb_local_begin", "bdg_cheb_local_read"):
        assert re.search(rf"^int {name}\(", header, flags=re.M)
        assert name in _native.SIGNATURES
    assert len(_native.SIGNATURES["bdg_cheb_local_begin"]) == 6
    assert len(_native.SIGNATURES["bdg_cheb_local_read"]) == 3
    for method in ("cheb_local_begin", "cheb_local_read"):
        assert callable(getattr(_native.System, method))
