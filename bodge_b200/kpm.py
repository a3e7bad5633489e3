"""Host-side post-processing of Chebyshev moments into observables.

The moments ``mu_n = <x|T_n(H/a)|x>`` come from the CUDA engine (``csrc/cheb.cu``); what is
left is O(n_moments) arithmetic per observable:

* free energy ``F = Tr g(H) = sum_n c_n mu_n`` with ``g(e) = -(T/2) ln(1 + exp(-e/T))``
  (``g(e) = min(e, 0)/2`` at T = 0), the trace form of the reference's
  ``bodge/hamiltonian.py:305-319``;
* resolvent diagonal ``<x|(z - H)^-1|x>`` for the LDOS of ``bodge/hamiltonian.py:349-382``.

No damping kernel is applied: ``g`` is analytic for T > 0 and the resolvent is evaluated off
the real axis, so the plain Chebyshev series converges geometrically (SURVEY 8c).
"""

from __future__ import annotations

import math

import numpy as np
from scipy.fft import dct
from scipy.special import expit


def free_energy_density(eps, temperature: float):
    """``g(eps)`` such that ``F = sum over ALL 4N eigenvalues of g``."""
    eps = np.asarray(eps, dtype=np.float64)
    if temperature < 0:
        raise ValueError("Expected non-negative temperature!")
    if temperature == 0:
        return np.minimum(eps, 0.0) / 2
    return -(temperature / 2) * np.logaddexp(0.0, -eps / temperature)


def chebyshev_coefficients(func, n_coef: int, scale: float) -> np.ndarray:
    """Coefficients ``c_n`` of ``x -> func(scale * x)`` in ``sum_n c_n T_n(x)`` by Chebyshev-Gauss
    quadrature on ``2 * n_coef`` nodes (a type-II DCT)."""
    nodes = 2 * n_coef
    theta = (np.arange(nodes) + 0.5) * (math.pi / nodes)
    samples = func(scale * np.cos(theta))
    coef = dct(samples, type=2)[:n_coef] / nodes
    coef[0] /= 2
    return coef


def fermi_coefficients(temperature: float, n_coef: int, scale: float) -> np.ndarray:
    """Coefficients ``c_n`` of the Fermi function ``f(ε) = 1/(1 + e^{ε/T})`` in ``f(scale * x) = sum_n c_n T_n(x)``, the
    series behind ``Hamiltonian.density_matrix``.  Like ``g`` of the free energy, ``f`` has its nearest poles at
    ``±iπT``, so ``free_energy_moments`` gives the length for a truncation error ``tol``.  T must be positive."""
    if not temperature > 0:
        raise ValueError("the Fermi function needs a temperature T > 0")
    return chebyshev_coefficients(lambda e: expit(-e / temperature), n_coef, scale)


def free_energy_from_trace(mu_trace, temperature: float, scale: float) -> float:
    """Free energy from the trace moments ``mu_n = Tr T_n(H / scale)``."""
    mu_trace = np.asarray(mu_trace, dtype=np.float64)
    coef = chebyshev_coefficients(lambda e: free_energy_density(e, temperature), len(mu_trace), scale)
    return float(coef @ mu_trace)


def default_moments(temperature: float, scale: float, tol: float = 1e-13, cap: int = 32768) -> int:
    """Series length for a smooth integrand: the coefficients of ``g`` decay like
    ``exp(-n * pi * T / scale)`` (nearest poles of the Fermi function at ``+-i pi T``)."""
    return free_energy_moments(temperature, scale, tol, cap)[0]


def free_energy_moments(temperature: float, scale: float, tol: float = 1e-13, cap: int = 32768) -> tuple[int, float]:
    """``(n, reached)``: series length for a relative truncation error ``tol`` of ``Tr g(H)`` and the error level
    actually reached with it.  T > 0: the coefficients decay like ``exp(-n pi T / scale)``; when the length that
    ``tol`` asks for exceeds ``cap`` the series stops there and ``reached = exp(-cap pi T / scale) > tol``.
    T = 0: ``g`` has a kink at the Fermi level, the coefficients decay only like ``1/n^2`` and ``reached`` is about
    ``(scale / n)^2``-limited -- 1e-7 relative at the default 8192 (measured, SURVEY 8c) -- whatever ``tol`` says."""
    if temperature <= 0:
        n = 8192 if cap >= 8192 else cap + (cap & 1)
        return n, 1e-7 * (8192 / n) ** 2
    rate = math.pi * temperature / scale
    n = int(math.ceil(-math.log(tol) / rate))
    reached = tol
    if n > cap:
        n, reached = cap, math.exp(-cap * rate)
    n = max(64, n)
    return n + (n & 1), reached


def resolvent_diagonal(mu, z: complex) -> complex:
    """``<x|(z - H~)^-1|x>`` from moments of ``H~`` for complex ``z`` off the real axis:
    ``(z - x)^-1 = (-i / sin t) sum_n (2 - delta_n0) T_n(x) exp(-i n t)``, ``t = arccos z`` taken
    on the branch where ``|exp(-i t)| < 1``."""
    mu = np.asarray(mu, dtype=np.float64)
    t = np.arccos(complex(z))
    if abs(np.exp(-1j * t)) > 1:
        t = -t
    w = np.exp(-1j * t)
    weights = 2.0 * mu
    weights[0] = mu[0]
    # Horner from the top keeps |w|^n factors from underflowing/overflowing.
    acc = 0j
    for m in weights[::-1]:
        acc = acc * w + m
    return (-1j / np.sin(t)) * acc


def resolvent_weights(z):
    """Per-energy constants of the resolvent series, vectorised over ``z``: ``w = exp(-i t)`` with
    ``t = arccos z`` on the branch where ``|w| < 1`` and the prefactor ``-i / sin t``, so that
    ``<x|(z - H~)^-1|x> = pref * sum_n (2 - delta_n0) mu_n w**n`` (the device kernel's inputs)."""
    z = np.asarray(z, dtype=np.complex128)
    t = np.arccos(z)
    t = np.where(np.abs(np.exp(-1j * t)) > 1, -t, t)
    return np.exp(-1j * t), -1j / np.sin(t)


def ldos_from_resolvent(g_imag, eps, energies) -> np.ndarray:
    """LDOS ``[site, energy]`` from ``Im <e_{4i+α}|(ε + iΓ - H)^-1|e_{4i+α}>`` given as
    ``g_imag[site, α, ε]`` for the sorted distinct ``eps = unique(|energies|)``: electrons
    (α = 0, 1) at ``+ε``, holes (α = 2, 3) at ``-ε`` (bodge/hamiltonian.py:376-382)."""
    energies = np.array(energies, dtype=float)
    pos = np.searchsorted(eps, np.abs(energies))
    electron = -(g_imag[:, 0, :] + g_imag[:, 1, :]) / math.pi
    hole = -(g_imag[:, 2, :] + g_imag[:, 3, :]) / math.pi
    # the reference fills ρ[+ε] then ρ[-ε] into one dict, so ε = 0 (being -0.0 == +0.0) ends up with the hole value
    use_electron = energies > 0
    return np.where(use_electron[None, :], electron[:, pos], hole[:, pos])


def ldos_moments_needed(scale: float, gamma_min: float, tol: float = 1e-13, cap: int = 1 << 20) -> int:
    """The resolvent series is geometric with ratio ``|exp(-i t)| ~ 1 - Γ/scale``."""
    return ldos_moments(scale, gamma_min, tol, cap)[0]


def ldos_moments(scale: float, gamma_min: float, tol: float = 1e-13, cap: int = 1 << 20) -> tuple[int, float]:
    """``(n, reached)`` like ``free_energy_moments``: length of the resolvent series for a truncation error ``tol``
    relative to its first term at broadening ``gamma_min``, and the level reached if ``cap`` cuts it short."""
    rate = gamma_min / scale
    n = int(math.ceil(-math.log(tol) / rate))
    reached = tol
    if n > cap:
        n, reached = cap, math.exp(-cap * rate)
    n = max(64, n)
    return n + (n & 1), reached


def series_error(n_moments: int, rate: float) -> float:
    """Truncation level ``exp(-n rate)`` of a geometric series cut after ``n_moments`` terms."""
    return math.exp(-min(n_moments * rate, 700.0))


def ldos_from_site_moments(mu4, energies, scale: float) -> np.ndarray:
    """LDOS at one site from the four unit-column moment series ``mu4[n, alpha]``.

    Follows the reference's conventions (bodge/hamiltonian.py:349-382): broadening
    ``Γ = np.gradient(unique(|ε|))`` per energy, electrons at ``+ε`` and holes at ``-ε``."""
    energies = np.array(energies, dtype=float)
    eps = np.unique(np.abs(energies))
    gamma = np.gradient(eps)
    table = {}
    for e, g in zip(eps, gamma):
        z = (e + 1j * g) / scale
        diag = [resolvent_diagonal(mu4[:, alpha], z) / scale for alpha in range(4)]
        table[+e] = -np.imag(diag[0] + diag[1]) / math.pi
        table[-e] = -np.imag(diag[2] + diag[3]) / math.pi
    return np.array([table[e] for e in energies])


# ------------------------------------------------------------------------------------------
# Spectral bounds from the moments (SURVEY 8f-4): Lanczos without a Lanczos kernel
# ------------------------------------------------------------------------------------------
def jacobi_from_moments(mu) -> tuple[np.ndarray, np.ndarray]:
    """Lanczos coefficients of ``(H~, x)`` from the Chebyshev moments ``mu_n = <x|T_n(H~)|x>``.

    The moments are the modified moments of the spectral measure of ``x`` with respect to the
    Chebyshev polynomials, so the modified Chebyshev algorithm (Sack-Donovan / Wheeler; Gautschi,
    *Orthogonal Polynomials*, 2.1.7) turns ``2m`` of them into the ``m x m`` Jacobi matrix that
    ``m`` Lanczos steps started at ``x`` would produce -- the GPU recursion that computes the
    moments IS the Krylov process, no extra kernel or vector pass is needed.  With the measure
    supported inside [-1, 1] the map is well conditioned.

    Returns ``(alpha[0..m-1], beta[1..m-1])``: diagonal and squared off-diagonal of the matrix.
    """
    nu = np.asarray(mu, dtype=np.float64)
    m = len(nu) // 2
    if m < 1 or nu[0] <= 0:
        raise ValueError("need at least two moments of a non-zero vector")
    # x T_l = a_l T_{l+1} + c_l T_{l-1}:  a_0 = 1, c_0 = 0;  a_l = c_l = 1/2 for l >= 1
    a = np.full(2 * m, 0.5)
    a[0] = 1.0
    c = np.full(2 * m, 0.5)
    c[0] = 0.0
    alpha, beta = np.zeros(m), np.zeros(m)
    alpha[0] = a[0] * nu[1] / nu[0]
    beta[0] = nu[0]
    prev2 = np.zeros(2 * m)   # sigma_{k-2, l}
    prev1 = nu[: 2 * m].copy()  # sigma_{k-1, l}
    for k in range(1, m):
        cur = np.zeros(2 * m)
        ls = np.arange(k, 2 * m - k)
        cur[ls] = a[ls] * prev1[ls + 1] - alpha[k - 1] * prev1[ls] + c[ls] * prev1[ls - 1] - beta[k - 1] * prev2[ls]
        if not cur[k] > 0:  # measure exhausted: the Krylov space is invariant after k steps
            return alpha[:k], beta[1:k]
        alpha[k] = a[k] * cur[k + 1] / cur[k] - a[k - 1] * prev1[k] / prev1[k - 1]
        beta[k] = a[k - 1] * cur[k] / prev1[k - 1]
        prev2, prev1 = prev1, cur
    return alpha, beta[1:]


def spectral_radius_from_moments(mu, scale: float) -> tuple[float, float]:
    """``(ritz, bound)`` for ``max |eigenvalue of H|`` from moments of ``H / scale``: the largest
    Ritz value in magnitude and the safeguarded estimate ``ritz + |residual|`` (the Ritz value
    approaches the spectral edge from inside; the residual of its Ritz vector bounds the distance to
    the nearest eigenvalue)."""
    from scipy.linalg import eigh_tridiagonal

    alpha, beta = jacobi_from_moments(mu)
    m = len(alpha)
    if m == 1:
        return abs(alpha[0]) * scale, abs(alpha[0]) * scale
    # keep the last coefficient as the residual norm of the (m-1)-step factorisation
    theta, vecs = eigh_tridiagonal(alpha[: m - 1], np.sqrt(beta[: m - 2])) if m > 2 else (alpha[:1], np.ones((1, 1)))
    k = int(np.argmax(np.abs(theta)))
    resid = math.sqrt(beta[m - 2]) * abs(vecs[-1, k])
    return float(abs(theta[k]) * scale), float((abs(theta[k]) + resid) * scale)
