"""CPU references for Fermi reads from distance-classed start columns (``Hamiltonian.density_matrix(spacing=...)``,
``bodge_b200.probing``) -- test infrastructure next to ``fermi_oracle.py``, with its conventions.

* ``polynomial_dense``: the dense truncated series ``P = Σ_{n < n_coef} c_n T_n(H/scale)`` of the Fermi function, the
  polynomial the GPU recursion applies;
* ``class_sum``: the prediction for a read from class columns, ``Σ_{j in class k} P[4i+α, 4j+β]``;
* ``class_local_kpm``: the scipy three-term recursion on the class columns themselves, accumulating the same reads as
  the GPU's local accumulator -- ``fermi_oracle.fermi_local_kpm`` with class indicators for unit columns."""

import numpy as np

import fermi_oracle as fo
from oracle import bdg_oracle as orc


def polynomial_dense(H, temperature, n_coef, scale):
    """``P = Σ_{n < n_coef} c_n T_n(H/scale)`` with the Chebyshev-Gauss coefficients of ``f(scale x)``, evaluated on
    the eigenvalues: ``U diag(p(ε/scale)) U^†`` (the same polynomial as the term-by-term sum, without its rounding)."""
    c = orc.cheb_coefficients(lambda e: fo.fermi(e, temperature), n_coef, scale)
    dense = H.toarray() if hasattr(H, "toarray") else np.asarray(H)
    eps, U = np.linalg.eigh(dense)
    return (U * np.polynomial.chebyshev.chebval(eps / scale, c)) @ U.conj().T


def class_columns(n_rows, site_class, class_rows):
    """``[n_rows, n_cols]`` start columns: column ``c`` is the indicator of class ``class_rows[c] >> 2`` in component
    ``class_rows[c] & 3``."""
    site_class = np.asarray(site_class)
    x = np.zeros((n_rows, len(class_rows)), dtype=np.complex128)
    for c, q in enumerate(np.asarray(class_rows, dtype=np.int64)):
        x[4 * np.flatnonzero(site_class == q >> 2) + (q & 3), c] = 1.0
    return x


def class_sum(P, site_class, class_rows, read_col, read_site):
    """``acc[r, α] = Σ_{j: class j = k} P[4 read_site[r] + α, 4j + β]`` with ``4k + β = class_rows[read_col[r]]``."""
    x = class_columns(P.shape[0], site_class, class_rows)
    Px = P @ x
    return Px[4 * np.asarray(read_site)[:, None] + np.arange(4), np.asarray(read_col)[:, None]]


def class_local_kpm(H, site_class, class_rows, read_col, read_site, temperature, n_coef, scale):
    """``acc[r, α] = Σ_n c_n (T_n(H/scale) x_{read_col[r]})[4 read_site[r] + α]`` by the three-term recursion."""
    c = orc.cheb_coefficients(lambda e: fo.fermi(e, temperature), n_coef, scale)
    Ht = H / scale
    idx = (4 * np.asarray(read_site)[:, None] + np.arange(4), np.asarray(read_col)[:, None])
    t_prev = class_columns(H.shape[0], site_class, class_rows)
    acc = c[0] * t_prev[idx]
    if n_coef == 1:
        return acc
    t_cur = Ht @ t_prev
    acc = acc + c[1] * t_cur[idx]
    for n in range(2, n_coef):
        t_prev, t_cur = t_cur, 2 * (Ht @ t_cur) - t_prev
        acc = acc + c[n] * t_cur[idx]
    return acc
