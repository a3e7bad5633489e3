"""Extended-precision light-cone reference of the Chebyshev recursion at any lattice size (test infrastructure).

A polynomial of degree ``n`` in ``H`` couples only sites within ``n`` hops.  So ``T_k(H~) x`` read at a site ``i``
depends only on ``x`` within ``k`` hops of ``i``, and the same recursion on a window of radius ``k`` around ``i`` with
open edges, the same blocks and ``x`` restricted to the window, gives it exactly.  For a probe column ``e_s`` the
whole ``T_k e_s`` is zero outside the ball of radius ``k`` around ``s``, so a window of radius ``n`` around ``s`` holds
``T_0 .. T_n`` in full.  A reference of a 10^7-site matrix then costs the size of the window.

* ``window``: the sites within ``r`` hops of the read sites, by breadth-first search over the cubic skeleton's stencil
  (wrap-around pairs included: the skeleton always has them, a non-wrapping axis stores zero blocks there).
* ``Lightcone.operator``: the window's blocks, read from the matrix the device holds (``System.lookup`` and
  ``System.gather_blocks``, or ``HostBlocks`` on the CPU), as the recursion of ``readout_cases.ScalarReference``
  (``np.longdouble`` when the matrix is real) or ``variant_cases.Reference``, with the library's float64 step factors.
  All-zero off-diagonal blocks are dropped, as ``eliminate_zeros`` does.
* Start vectors restricted to the window: probe rows, Rademacher columns at global rows (``rademacher_rows``), class
  columns (``class_start``).
* ``run_probes``: ``T_{n-1}`` and ``T_n`` of probe columns in full (window rows mapped back to global rows) and their
  moments ``mu_0 .. mu_{2n-1}`` from ``mu_2k = 2 <T_k,T_k> - mu_0``, ``mu_2k+1 = 2 <T_k+1,T_k> - mu_1``, which is what a
  recursion at ``T_n`` has.  ``run_reads``: ``T_k`` at read sites for any start vector.

The window recursions are independent jobs: ``Lightcone.solve`` spreads them over host processes.
"""

from __future__ import annotations

import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor
from dataclasses import dataclass

import numpy as np

from oracle import bdg_oracle as orc


# ---- windows --------------------------------------------------------------------------------------------------------
def coords(shape, flat):
    """``(x, y, z)`` of flat indices ``z + Lz*(y + Ly*x)``."""
    flat = np.asarray(flat, dtype=np.int64)
    _, Ly, Lz = shape
    return flat // (Ly * Lz), (flat // Lz) % Ly, flat % Lz


def neighbours(shape, flat):
    """``[len(flat), m]`` stencil neighbours: ``x +- 1`` modulo the length along every axis of length >= 2 (on a
    two-site axis both are the same site)."""
    flat = np.asarray(flat, dtype=np.int64)
    c = coords(shape, flat)
    strides = (shape[1] * shape[2], shape[2], 1)
    out = []
    for axis, L in enumerate(shape):
        if L < 2:
            continue
        for d in (1, -1):
            out.append(flat + ((c[axis] + d) % L - c[axis]) * strides[axis])
    return np.stack(out, axis=1) if out else np.empty((len(flat), 0), dtype=np.int64)


def window(shape, sites, radius):
    """Sorted flat indices of the sites within ``radius`` hops of ``sites`` (breadth-first search)."""
    seen = np.unique(np.asarray(sites, dtype=np.int64))
    frontier = seen
    for _ in range(int(radius)):
        if frontier.size == 0:
            break
        reach = np.unique(neighbours(shape, frontier))
        frontier = np.setdiff1d(reach, seen, assume_unique=True)
        seen = np.union1d(seen, frontier)
    return seen


def local_index(win, flat):
    """Window positions of flat indices (all must lie in the window)."""
    flat = np.asarray(flat, dtype=np.int64)
    pos = np.searchsorted(win, flat)
    assert np.all(pos < len(win)) and np.array_equal(win[np.minimum(pos, len(win) - 1)], flat), "site outside the window"
    return pos


def scalar_rows(sites):
    """The scalar rows ``4 i + alpha`` of ``sites``, site-major."""
    return (4 * np.asarray(sites, dtype=np.int64)[:, None] + np.arange(4)).ravel()


# ---- start vectors at global rows ------------------------------------------------------------------------------------
def rademacher_rows(seed, rows, cols):
    """``orc.rademacher(seed, ., cols)`` at the global scalar ``rows`` only: the same counter hash, evaluated at ``rows``."""
    u = orc.U64
    rows = np.asarray(rows, dtype=u)
    cols = np.asarray(cols, dtype=u)
    with np.errstate(over="ignore"):
        hc = orc._mix64(u(seed) + orc._GAMMA * (cols + u(1)))
        h = orc._mix64(hc[None, :] + orc._GAMMA * (rows[:, None] + u(1)))
    return np.where(h >> u(63), -1.0, 1.0).astype(np.complex128)


def class_start(site_class, rows, class_rows):
    """Class columns ``4k + beta`` (``BDG_X0_CLASS``) at the global scalar ``rows``: 1 where the row's site is of class
    ``k`` and its component is ``beta``."""
    rows = np.asarray(rows, dtype=np.int64)
    class_rows = np.asarray(class_rows, dtype=np.int64)
    cls = np.asarray(site_class)[rows // 4]
    hit = (cls[:, None] == class_rows[None, :] // 4) & ((rows % 4)[:, None] == class_rows[None, :] % 4)
    return hit.astype(np.complex128)


def probe_start(rows, probe_rows):
    return (np.asarray(rows, dtype=np.int64)[:, None] == np.asarray(probe_rows, dtype=np.int64)[None, :]).astype(np.complex128)


# ---- blocks ----------------------------------------------------------------------------------------------------------
class HostBlocks:
    """Host stand-in for ``System.lookup`` / ``System.gather_blocks`` over skeleton arrays (``indptr``, ``indices``,
    ``data`` with every skeleton block, zero or not)."""

    def __init__(self, indptr, indices, data):
        self.indptr, self.indices, self.data = np.asarray(indptr), np.asarray(indices), np.asarray(data)

    def lookup(self, i, j):
        return orc.block_index(self.indptr, self.indices, i, j)

    def gather_blocks(self, k):
        return self.data[np.asarray(k, dtype=np.int64)].copy()


def window_bsr(shape, win, source):
    """BSR arrays of the matrix restricted to the window ``win`` (open edges), columns in window positions, blocks in
    ascending column order; all-zero off-diagonal blocks dropped, the diagonal block always kept."""
    n = len(win)
    cand = np.concatenate([win[:, None], neighbours(shape, win)], axis=1)
    cand.sort(axis=1)
    keep = np.ones(cand.shape, dtype=bool)
    keep[:, 1:] = cand[:, 1:] != cand[:, :-1]          # a two-site axis lists its one neighbour twice
    pos = np.searchsorted(win, cand)
    keep &= (pos < n) & (win[np.minimum(pos, n - 1)] == cand)
    row = np.broadcast_to(np.arange(n)[:, None], cand.shape)[keep]
    gi, gj = win[row], cand[keep]
    blocks = source.gather_blocks(source.lookup(gi, gj))
    nz = np.any(blocks != 0, axis=(1, 2)) | (gi == gj)
    row, col, blocks = row[nz], pos[keep][nz], blocks[nz]
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(row, minlength=n), out=indptr[1:])
    return indptr, col.astype(np.int64), blocks


def operator(indptr, indices, data, scale):
    """``ScalarReference`` when every scalar row keeps a non-zero, else the block ``Reference``."""
    from readout_cases import ScalarReference
    from variant_cases import Reference

    try:
        return ScalarReference(indptr, indices, data, scale)
    except AssertionError:
        return Reference(indptr, indices, data, scale)


def _start(ref, x0):
    x0 = np.asarray(x0)
    if hasattr(ref, "start"):
        return ref.start(x0)
    return x0.astype(np.clongdouble)


# ---- jobs (run in worker processes: numpy only, no device) -------------------------------------------------------------
@dataclass
class Job:
    """One window recursion: the window's BSR arrays, the start block ``x0`` (``[4 n_w, C]``), the number of steps and
    what to keep: ``moments`` (``mu_0 .. mu_{2n-1}``), ``full`` (T_{n-1} and T_n), ``reads`` (``{k: window scalar rows
    [R, 4] and their columns [R]}``)."""
    indptr: np.ndarray
    indices: np.ndarray
    data: np.ndarray
    scale: float
    x0: np.ndarray
    n: int
    moments: bool = False
    full: bool = False
    read_rows: np.ndarray | None = None   # [R, 4] window scalar rows
    read_cols: np.ndarray | None = None   # [R] columns of x0
    read_ks: tuple = ()


def run_job(job: Job):
    ref = operator(job.indptr, job.indices, job.data, job.scale)
    x = _start(ref, job.x0)
    mu = np.zeros((2 * job.n, x.shape[1]), dtype=np.longdouble) if job.moments else None
    reads = {}
    prev, cur = None, x
    mu0 = mu1 = None
    for k in range(job.n + 1):
        if k == 1:
            prev, cur = cur, ref.a1 * ref.matvec(cur)
        elif k >= 2:
            prev, cur = cur, ref.a2 * ref.matvec(cur) - prev
        if mu is not None:
            if k == 0:
                mu0 = (x.conj() * x).sum(axis=0).real
                mu[0] = mu0
            elif k == 1:
                mu1 = (x.conj() * cur).sum(axis=0).real
                mu[1] = mu1
            if 1 <= k < job.n:
                mu[2 * k] = 2 * (cur.conj() * cur).sum(axis=0).real - mu0
            if k >= 2:
                mu[2 * k - 1] = 2 * (cur.conj() * prev).sum(axis=0).real - mu1
        if k in job.read_ks:
            reads[k] = cur[job.read_rows, job.read_cols[:, None]].astype(np.clongdouble)
    full = (prev if job.n >= 1 else None, cur) if job.full else None
    return mu, full, reads


def solve(jobs, workers=None):
    """``run_job`` over ``jobs``, in worker processes when ``workers`` (default: the host cores) is more than one."""
    workers = min(len(jobs), workers or os.cpu_count() or 1)
    if workers <= 1:
        return [run_job(j) for j in jobs]
    with ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("spawn")) as pool:
        return list(pool.map(run_job, jobs))


# ---- the reference -------------------------------------------------------------------------------------------------------
class Lightcone:
    """Window references of the recursion on ``H / scale`` of a ``CubicLattice(shape)`` matrix whose blocks ``source``
    supplies (a ``System`` or ``HostBlocks``)."""

    def __init__(self, shape, source, scale):
        self.shape = tuple(int(v) for v in shape)
        self.n_sites = int(np.prod(self.shape))
        self.source = source
        self.scale = float(scale)

    def probe_jobs(self, probe_rows, n):
        """One job per probe site, on a window of radius ``n`` around it; returns ``(jobs, windows, columns per job)``."""
        probe_rows = np.asarray(probe_rows, dtype=np.int64)
        jobs, wins, groups = [], [], []
        for s in np.unique(probe_rows // 4):
            cols = np.flatnonzero(probe_rows // 4 == s)
            win = window(self.shape, [s], n)
            x0 = probe_start(scalar_rows(win), probe_rows[cols])
            jobs.append(Job(*window_bsr(self.shape, win, self.source), self.scale, x0, n, moments=True, full=True))
            wins.append(win)
            groups.append(cols)
        return jobs, wins, groups

    def run_probes(self, probe_rows, n, workers=None):
        """Probe columns ``e_r``: ``(mu [2n, C] longdouble, vectors)``; ``vectors[c] = (global scalar rows, T_{n-1} there,
        T_n there)`` (clongdouble / longdouble), zero at every other row."""
        jobs, wins, groups = self.probe_jobs(probe_rows, n)
        mu = np.zeros((2 * n, len(probe_rows)), dtype=np.longdouble)
        vectors = [None] * len(probe_rows)
        for (m, (prev, cur), _), win, cols in zip(solve(jobs, workers), wins, groups):
            mu[:, cols] = m
            rows = scalar_rows(win)
            for j, c in enumerate(cols):
                vectors[c] = (rows, prev[:, j], cur[:, j])
        return mu, vectors

    def read_jobs(self, start, cols, sites, ks):
        """One job per distinct column: the window of radius ``max(ks)`` around that column's read sites."""
        cols, sites = np.asarray(cols, dtype=np.int64), np.asarray(sites, dtype=np.int64)
        radius = max(ks)
        jobs, groups = [], []
        for c in np.unique(cols):
            idx = np.flatnonzero(cols == c)
            win = window(self.shape, sites[idx], radius)
            x0 = start(scalar_rows(win), [c])
            rows = 4 * local_index(win, sites[idx])[:, None] + np.arange(4)
            jobs.append(Job(*window_bsr(self.shape, win, self.source), self.scale, x0, radius, read_rows=rows,
                            read_cols=np.zeros(len(idx), dtype=np.int64), read_ks=tuple(ks)))
            groups.append(idx)
        return jobs, groups

    def run_reads(self, start, cols, sites, ks, workers=None):
        """``T_k[4 sites[r] + alpha, cols[r]]`` as ``{k: [R, 4] clongdouble}`` for start columns ``start(rows, cols)``
        (global scalar rows, global column ids) -- e.g. ``rademacher_rows`` or ``class_start`` bound to their data."""
        jobs, groups = self.read_jobs(start, cols, sites, ks)
        out = {k: np.zeros((len(sites), 4), dtype=np.clongdouble) for k in ks}
        for (_, _, reads), idx in zip(solve(jobs, workers), groups):
            for k in ks:
                out[k][idx] = reads[k]
        return out
