"""Extended-precision references of the Chebyshev read-outs: the moments, the resolvent series behind ``ldos``, the series
contraction behind ``free_energy`` and the local sums behind ``density_matrix``.

Everything is computed from the ``np.clongdouble`` vectors of ``variant_cases.Reference`` by the definitions, without
the moment doubling or the even-vector identities the device uses, so that a read-out can be checked moment by moment
at the recursion lengths the observables run.  ``test_readout_cases.py`` pins these helpers against the float64
oracle; ``test_gpu_readout.py`` checks the device against them.
"""

from __future__ import annotations

import numpy as np

EPS = np.finfo(np.float64).eps


class ScalarReference:
    """``variant_cases.Reference`` over the scalar non-zeros of the same BSR arrays: the same recursion in extended
    precision, an order of magnitude faster on the sparse 4x4 blocks of BdG models, and in ``np.longdouble`` alone when
    the matrix is real (real start vectors then keep every ``T_n`` real).  Long references (10^5 steps) need that."""

    def __init__(self, indptr, indices, data, scale):
        from variant_cases import longdouble_check

        longdouble_check()
        indptr, indices, data = np.asarray(indptr), np.asarray(indices), np.asarray(data)
        n = len(indptr) - 1
        brow = np.repeat(np.arange(n), np.diff(indptr))
        rows = np.broadcast_to(4 * brow[:, None, None] + np.arange(4)[None, :, None], data.shape).ravel()
        cols = np.broadcast_to(4 * indices[:, None, None] + np.arange(4)[None, None, :], data.shape).ravel()
        vals = data.ravel()
        keep = vals != 0
        rows, cols, vals = rows[keep], cols[keep], vals[keep]
        order = np.lexsort((cols, rows))
        rows, self.cols, vals = rows[order], cols[order], vals[order]
        assert np.array_equal(np.unique(rows), np.arange(4 * n)), "every scalar row needs a non-zero (reduceat)"
        self.starts = np.searchsorted(rows, np.arange(4 * n))
        self.real = not np.any(vals.imag)
        self.vals = (vals.real.astype(np.longdouble) if self.real else vals.astype(np.clongdouble))[:, None]
        self.a1 = np.longdouble(1.0 / scale)
        self.a2 = np.longdouble(2.0 / scale)

    def start(self, x0):
        """``x0`` in the working type: longdouble when both the matrix and ``x0`` are real."""
        x0 = np.asarray(x0)
        if self.real and not np.any(x0.imag):
            return x0.real.astype(np.longdouble)
        return x0.astype(np.clongdouble)

    def matvec(self, x):
        return np.add.reduceat(self.vals * x[self.cols], self.starts, axis=0)


def reference_readouts(ref, x0, n_moments, local=None):
    """``mu[n, c] = Re <x_c|T_n x_c>`` for ``n < n_moments`` in ``np.longdouble``, one clongdouble vector per moment.

    ``local = (rows, cols, n_terms)``: also ``T_n[rows[r], cols[r]]`` for ``n < n_terms`` as ``[n_terms, len(rows)]``
    clongdouble (the terms of the local sums).  Returns ``(mu, terms, t_max)``: ``terms`` is None without ``local``,
    ``t_max`` the largest ``|T_n|`` entry of the local terms' vectors (``n < n_terms``), 0 without ``local``."""
    x = ref.start(x0) if hasattr(ref, "start") else np.asarray(x0).astype(np.clongdouble)
    xc = x.conj()
    mu = np.empty((n_moments, x.shape[1]), dtype=np.longdouble)
    terms = None
    if local is not None:
        rows, cols, n_terms = local
        rows, cols = np.asarray(rows), np.asarray(cols)
        terms = np.empty((n_terms, len(rows)), dtype=np.clongdouble)
    else:
        n_terms = 0
    prev, cur = None, x
    t_max = 0.0
    for n in range(max(n_moments, n_terms)):
        if n == 1:
            prev, cur = cur, ref.a1 * ref.matvec(cur)
        elif n >= 2:
            prev, cur = cur, ref.a2 * ref.matvec(cur) - prev
        if n < n_moments:
            mu[n] = (xc * cur).sum(axis=0).real
        if n < n_terms:
            terms[n] = cur[rows, cols]
            t_max = max(t_max, float(np.max(np.abs(cur))))
    return mu, terms, t_max


def resolvent(mu, w, pref):
    """``g[c, e] = pref[e] sum_n (2 - delta_n0) mu[n, c] w[e]^n`` in clongdouble from the float64 ``w`` and ``pref`` the
    device receives, and ``sum_n |(2 - delta_n0) mu[n, c] w[e]^n| |pref[e]|``, the scale its rounding is measured on.
    ``mu``: ``[n_moments, n_cols]``."""
    mu = np.asarray(mu).astype(np.longdouble)
    w = np.asarray(w).astype(np.clongdouble)
    pref = np.asarray(pref).astype(np.clongdouble)
    acc = np.zeros((mu.shape[1], len(w)), dtype=np.clongdouble)
    size = np.zeros((mu.shape[1], len(w)), dtype=np.longdouble)
    aw = np.abs(w)
    for n in range(mu.shape[0] - 1, -1, -1):
        m = (1 if n == 0 else 2) * mu[n][:, None]
        acc = acc * w[None, :] + m
        size = size * aw[None, :] + np.abs(m)
    return acc * pref[None, :], size * np.abs(pref)[None, :]


def contract(mu, coef):
    """``out[c] = sum_n coef[n] mu[n, c]`` in longdouble, and ``sum_n |coef[n] mu[n, c]|``."""
    mu = np.asarray(mu).astype(np.longdouble)
    coef = np.asarray(coef).astype(np.longdouble)[:, None]
    return (coef * mu).sum(axis=0), np.abs(coef * mu).sum(axis=0)


def local_sums(terms, coef):
    """``sum_n coef[n] T_n[row_r, col_r]`` from the ``terms`` of ``reference_readouts``, and ``sum_n |coef[n]| |T_n|``."""
    coef = np.asarray(coef).astype(np.longdouble)[:, None]
    terms = terms[: len(coef)]
    return (coef * terms).sum(axis=0), (np.abs(coef) * np.abs(terms)).sum(axis=0)


def warp_sum(values):
    """The float64 sum of ``values`` in the order of the one-warp reduction of ``observables.cu`` (``sum_columns``):
    lane ``l`` adds ``values[l], values[l + 32], ...`` in turn, then an xor butterfly over 16, 8, 4, 2, 1 lanes."""
    values = np.asarray(values, dtype=np.float64)
    lanes = np.zeros(32)
    for i, v in enumerate(values):
        lanes[i % 32] += v
    for d in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[np.arange(32) ^ d]
    return float(lanes[0])


def moment_ratios(got, want):
    """``|got[n, c] - want[n, c]| / ((n + 1) eps64 mu_0[c])``, per moment and column (``mu_0 = |x_c|^2 > 0``)."""
    got = np.asarray(got).astype(np.longdouble)
    want = np.asarray(want)
    n = np.arange(want.shape[0], dtype=np.longdouble)[:, None]
    return np.abs(got - want) / ((n + 1) * EPS * want[0][None, :])


def worst(ratios, parity=None):
    """The largest of ``ratios`` (``[n, c]``), over the even (``parity=0``) or odd (``1``) moments only, as a float."""
    r = ratios if parity is None else ratios[parity::2]
    return float(np.max(r)) if r.size else 0.0


def random_hermitian_bsr(shape, seed):
    """A Hermitian BSR matrix on the nearest-neighbour skeleton of a cubic ``shape``, with random complex blocks, and
    an upper bound of its spectral radius (its infinity norm)."""
    from oracle import bdg_oracle as orc

    indptr, indices = orc.cubic_skeleton(shape)
    rng = np.random.default_rng(seed)
    n = len(indptr) - 1
    data = np.zeros((len(indices), 4, 4), dtype=np.complex128)
    for i in range(n):
        for p in range(indptr[i], indptr[i + 1]):
            j = int(indices[p])
            if j < i:
                continue
            b = rng.standard_normal((4, 4)) + 1j * rng.standard_normal((4, 4))
            if j == i:
                b = b + b.conj().T
            data[p] = b
            if j != i:
                q = indptr[j] + int(np.searchsorted(indices[indptr[j]:indptr[j + 1]], i))
                data[q] = b.conj().T
    return indptr, indices, data, orc.norm_inf(indptr, indices, data)
