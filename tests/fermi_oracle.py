"""CPU references for the local density matrix ``ρ = f(H)``, ``f(ε) = 1/(1 + e^{ε/T})`` -- test infrastructure, like
``oracle/bdg_oracle.py`` whose matrices and recursion conventions it uses.

* ``fermi_dense``: the exact ``f(H)`` of a dense matrix by ``eigh``;
* ``fermi_local_kpm``: the Chebyshev series of ``f`` on probe columns by the scipy three-term recursion, accumulating
  the same reads as the GPU's local accumulator (``bdg_cheb_local_begin``);
* ``gap_fixed_point``: the plain fixed-point iteration ``Δ_i = -V ρ[4i, 4i+3]`` of the s-wave gap equation, dense.

The reference has no such code (its only route to ``ρ`` is ``diagonalize()``); the sign convention is pinned to the
reference's own free energy by the Hellmann-Feynman test in ``test_density_oracle.py``."""

import numpy as np
from scipy.special import expit

from oracle import bdg_oracle as orc


def fermi(eps, temperature):
    return expit(-np.asarray(eps, dtype=float) / temperature)


def fermi_dense(H_dense, temperature):
    """``f(H) = U diag(f(ε)) U^†`` from ``numpy.linalg.eigh``."""
    eps, U = np.linalg.eigh(np.asarray(H_dense))
    return (U * fermi(eps, temperature)) @ U.conj().T


def fermi_local_kpm(H, rows, read_col, read_site, temperature, n_coef, scale):
    """``acc[r, α] = Σ_{n < n_coef} c_n T_n(H/scale)[4 read_site[r] + α, rows[read_col[r]]]`` with ``c_n`` the
    Chebyshev-Gauss coefficients of ``f(scale x)``: one SpMM per term on the probe columns ``e_rows``."""
    c = orc.cheb_coefficients(lambda e: fermi(e, temperature), n_coef, scale)
    Ht = H / scale
    idx = (4 * np.asarray(read_site)[:, None] + np.arange(4), np.asarray(read_col)[:, None])
    t_prev = orc.probes(H.shape[0], rows)
    acc = c[0] * t_prev[idx]
    if n_coef == 1:
        return acc
    t_cur = Ht @ t_prev
    acc = acc + c[1] * t_cur[idx]
    for n in range(2, n_coef):
        t_prev, t_cur = t_cur, 2 * (Ht @ t_cur) - t_prev
        acc = acc + c[n] * t_cur[idx]
    return acc


def square_attractive(L, delta, mu=-1.0, t=1.0):
    """Dense ``H`` of an open ``L x L`` lattice: ``H[i,i] = -μ σ0``, bonds ``-t σ0``, ``Δ[i,i] = Δ_i jσ2``
    (the site order of ``CubicLattice((L, L, 1))``)."""
    N = L * L
    s0, js2 = np.eye(2), np.array([[0.0, 1.0], [-1.0, 0.0]])
    M = np.zeros((4 * N, 4 * N), dtype=np.complex128)
    for x in range(L):
        for y in range(L):
            i = x * L + y
            M[4 * i:4 * i + 2, 4 * i:4 * i + 2] = -mu * s0
            M[4 * i + 2:4 * i + 4, 4 * i + 2:4 * i + 4] = mu * s0
            M[4 * i:4 * i + 2, 4 * i + 2:4 * i + 4] = delta[i] * js2
            M[4 * i + 2:4 * i + 4, 4 * i:4 * i + 2] = (delta[i] * js2).conj().T
            for X, Y in ((x + 1, y), (x - 1, y), (x, y + 1), (x, y - 1)):
                if 0 <= X < L and 0 <= Y < L:
                    j = X * L + Y
                    M[4 * i:4 * i + 2, 4 * j:4 * j + 2] = -t * s0
                    M[4 * i + 2:4 * i + 4, 4 * j + 2:4 * j + 4] = t * s0
    return M


def gap_fixed_point(L, V, temperature, start=0.1, tol=1e-12, max_iter=1000, **model):
    """Plain iteration ``Δ_i <- -V f(H(Δ))[4i, 4i+3]`` from ``Δ_i = start`` until ``max|ΔΔ| <= tol``: ``(Δ, iterations)``."""
    N = L * L
    delta = np.full(N, start, dtype=np.complex128)
    d = 4 * np.arange(N)
    for it in range(1, max_iter + 1):
        new = -V * fermi_dense(square_attractive(L, delta, **model), temperature)[d, d + 3]
        step = np.max(np.abs(new - delta))
        delta = new
        if step <= tol:
            return delta, it
    raise RuntimeError("gap_fixed_point did not converge")
