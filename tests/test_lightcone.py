"""The light-cone reference of ``lightcone.py`` against the full-lattice extended-precision recursion (CPU only).

On small lattices the whole-lattice recursion is cheap.  The window results must equal it.  The window's rows keep the
scalar entries of the lattice's rows in the same order, but a row at the window's rim has fewer of them, and numpy sums
a row of eight or more terms in eight partial sums: there ``T_k`` may differ in the last bits of ``np.longdouble``, and
nowhere else.  When the window is the whole lattice, ``T_k`` must be the same bits.  The moments, taken by doubling here
and by definition there, agree to the rounding of ``np.longdouble``.  Lattices: open, wrapping and mixed axes in
1-D, 2-D and 3-D, cones that reach an open edge, that cross a wrap seam, and that are wider than the lattice.  The
blocks come from ``HostBlocks``, the host stand-in for ``System.lookup`` / ``System.gather_blocks``.
"""

import numpy as np
import pytest

import lightcone as lc
import readout_cases as rc
from bodge_b200 import probing
from oracle import bdg_oracle as orc

EPS_LD = float(np.finfo(np.longdouble).eps)

# name: (shape, wrapping axes)
LATTICES = {
    "chain_open": ((23, 1, 1), (False, False, False)),
    "chain_ring": ((23, 1, 1), (True, False, False)),
    "plane_mixed": ((11, 8, 1), (True, False, False)),
    "plane_torus": ((7, 9, 1), (True, True, False)),
    "plane_two_site": ((2, 10, 1), (False, True, False)),
    "cube_mixed": ((5, 4, 6), (False, True, True)),
    "cube_open": ((4, 5, 3), (False, False, False)),
}


def hermitian(shape, wraps, seed=3, real=False):
    """Skeleton arrays with random Hermitian blocks; the edge blocks of axes that do not wrap are zero."""
    indptr, indices, data, norm = rc.random_hermitian_bsr(shape, seed)
    if real:
        data = data.real.astype(np.complex128)
    for axis, L in enumerate(shape):
        if L >= 3 and not wraps[axis]:
            idx = np.arange(int(np.prod(shape))).reshape(shape)
            lo, hi = np.take(idx, 0, axis=axis).ravel(), np.take(idx, L - 1, axis=axis).ravel()
            k = orc.block_index(indptr, indices, np.concatenate([lo, hi]), np.concatenate([hi, lo]))
            data[k] = 0
    return indptr, indices, data, 1.01 * norm


def ld_ratio(got, want, k):
    """``max|got - want| / ((k + 1) eps_longdouble max(1, max|want|))``: the rounding of a different summation order in
    ``np.longdouble`` keeps it small; 0 for the same bits."""
    err = float(np.max(np.abs(np.asarray(got) - np.asarray(want)))) if np.size(want) else 0.0
    return err / ((k + 1) * EPS_LD * max(1.0, float(np.max(np.abs(want)))))


def full_vectors(indptr, indices, data, scale, x0, n):
    ref = rc.ScalarReference(indptr, indices, data, scale)
    out = [ref.start(x0)]
    if n >= 1:
        out.append(ref.a1 * ref.matvec(out[0]))
    for _ in range(2, n + 1):
        out.append(ref.a2 * ref.matvec(out[-1]) - out[-2])
    return out


def torus_distance(shape, a, b):
    ca, cb = lc.coords(shape, a), lc.coords(shape, b)
    d = 0
    for axis, L in enumerate(shape):
        dx = np.abs(ca[axis] - cb[axis])
        d = d + np.minimum(dx, L - dx)
    return d


def sites_of(shape):
    """A corner, the far corner, a site next to the x seam and one in the middle."""
    n = int(np.prod(shape))
    Lx, Ly, Lz = shape
    return sorted({0, n - 1, (Lx - 1) * Ly * Lz + (Ly // 2) * Lz, n // 2})


@pytest.mark.parametrize("name", list(LATTICES))
@pytest.mark.parametrize("radius", [0, 1, 3, 6, 40])
def test_window_is_the_ball_of_the_skeleton_stencil(name, radius):
    shape, _ = LATTICES[name]
    n = int(np.prod(shape))
    sites = sites_of(shape)[:2]
    want = np.flatnonzero(np.min([torus_distance(shape, np.arange(n), s) for s in sites], axis=0) <= radius)
    win = lc.window(shape, sites, radius)
    assert np.array_equal(win, want)
    assert np.array_equal(lc.local_index(win, win), np.arange(len(win)))
    if radius >= sum(shape):
        assert len(win) == n  # a cone wider than the lattice covers it


def test_rademacher_rows_are_the_oracle_rows():
    want = orc.rademacher(77, 4 * 300, np.arange(3, 9))
    rows = np.array([0, 1, 5, 123, 1199])
    assert np.array_equal(lc.rademacher_rows(77, rows, np.arange(3, 9)), want[rows])


@pytest.mark.parametrize("name", list(LATTICES))
@pytest.mark.parametrize("n", [1, 4, 9, 30])
def test_probe_columns_equal_the_full_recursion(name, n):
    shape, wraps = LATTICES[name]
    indptr, indices, data, scale = hermitian(shape, wraps, real=name == "cube_open")
    cone = lc.Lightcone(shape, lc.HostBlocks(indptr, indices, data), scale)
    sites = sites_of(shape)
    probe_rows = np.array([4 * s + b for s in sites for b in (0, 3)] + [4 * sites[0] + 2])
    mu, vectors = cone.run_probes(probe_rows, n, workers=1)

    N = int(np.prod(shape))
    x0 = orc.probes(4 * N, probe_rows)
    full = full_vectors(indptr, indices, data, scale, x0, n)
    for c, (rows, prev, cur) in enumerate(vectors):
        for k, got, want in ((n, cur, full[n][:, c]), (n - 1, prev, full[n - 1][:, c])):
            dense = np.zeros(4 * N, dtype=want.dtype)
            dense[rows] = got
            if len(rows) == 4 * N:
                assert np.array_equal(dense, want), f"column {c}: T_{k} on a window that is the lattice"
            assert ld_ratio(dense, want, k) <= 64, f"column {c}: the window's T_{k} differs from the lattice's"
    want_mu = rc.reference_readouts(rc.ScalarReference(indptr, indices, data, scale), x0, 2 * n)[0]
    m = np.arange(2 * n)[:, None]
    assert np.all(np.abs(mu - want_mu) <= 64 * (m + 1) * EPS_LD * want_mu[0])


@pytest.mark.parametrize("name", list(LATTICES))
@pytest.mark.parametrize("start", ["rademacher", "class"])
def test_reads_of_any_start_vector_equal_the_full_recursion(name, start):
    shape, wraps = LATTICES[name]
    indptr, indices, data, scale = hermitian(shape, wraps, seed=8)
    cone = lc.Lightcone(shape, lc.HostBlocks(indptr, indices, data), scale)
    N = int(np.prod(shape))
    all_rows = np.arange(4 * N)
    if start == "rademacher":
        n_cols = 3
        fn = lambda rows, cols: lc.rademacher_rows(41, rows, cols)  # noqa: E731
    else:
        site_class, n_classes = probing.site_classes(shape, 3, wraps)
        class_rows = np.array([4 * int(site_class[s]) + b for s, b in ((0, 1), (N - 1, 0), (N // 2, 3))])
        n_cols = len(class_rows)
        fn = lambda rows, cols: lc.class_start(site_class, rows, class_rows[np.asarray(cols)])  # noqa: E731
    sites = np.array(sites_of(shape) * n_cols)
    cols = np.repeat(np.arange(n_cols), len(sites_of(shape)))
    ks = (0, 1, 2, 5, 8)
    got = cone.run_reads(fn, cols, sites, ks, workers=1)
    full = full_vectors(indptr, indices, data, scale, fn(all_rows, np.arange(n_cols)), max(ks))
    for k in ks:
        want = full[k][4 * sites[:, None] + np.arange(4), cols[:, None]]
        assert ld_ratio(got[k], want, k) <= 64, f"T_{k} at the read sites"


def _perturbed(data, indptr, indices, site):
    out = data.copy()
    k = orc.block_index(indptr, indices, [site], [site])[0]
    out[k] = out[k] + 1e-3 * np.diag([1.0, -1.0, 1.0, -1.0])
    return out


@pytest.mark.parametrize("name", ["plane_torus", "cube_mixed", "chain_open"])
def test_a_block_outside_the_cone_leaves_it_and_one_inside_changes_it(name):
    shape, wraps = LATTICES[name]
    indptr, indices, data, scale = hermitian(shape, wraps)
    N = int(np.prod(shape))
    n, s = 3, 0
    dist = torus_distance(shape, np.arange(N), s)
    rows = np.array([4 * s, 4 * s + 1])
    base = lc.Lightcone(shape, lc.HostBlocks(indptr, indices, data), scale).run_probes(rows, n, workers=1)
    far = int(np.flatnonzero(dist == n + 1)[0])
    near = int(np.flatnonzero(dist == n - 1)[0])
    for site, same in ((far, True), (near, False)):
        other = lc.Lightcone(shape, lc.HostBlocks(indptr, indices, _perturbed(data, indptr, indices, site)), scale)
        mu, vectors = other.run_probes(rows, n, workers=1)
        equal = np.array_equal(mu, base[0]) and all(np.array_equal(a[2], b[2]) for a, b in zip(vectors, base[1]))
        assert equal == same, f"block at distance {dist[site]} from the probe"


def test_a_window_one_hop_short_is_seen():
    """The comparison of ``test_probe_columns_equal_the_full_recursion`` sees a window of radius n - 1: T_n at the cone's
    rim is lost."""
    shape, wraps = LATTICES["plane_torus"]
    indptr, indices, data, scale = hermitian(shape, wraps)
    cone = lc.Lightcone(shape, lc.HostBlocks(indptr, indices, data), scale)
    n, s = 3, 5
    win = lc.window(shape, [s], n - 1)
    x0 = lc.probe_start(lc.scalar_rows(win), [4 * s])
    job = lc.Job(*lc.window_bsr(shape, win, cone.source), scale, x0, n, full=True)
    _, (_, cur), _ = lc.run_job(job)
    N = int(np.prod(shape))
    want = full_vectors(indptr, indices, data, scale, orc.probes(4 * N, [4 * s]), n)[n][:, 0]
    dense = np.zeros(4 * N, dtype=want.dtype)
    dense[lc.scalar_rows(win)] = cur[:, 0]
    assert ld_ratio(dense, want, n) > 1e6


def test_worker_processes_give_the_same_bits():
    shape, wraps = LATTICES["plane_torus"]
    indptr, indices, data, scale = hermitian(shape, wraps)
    cone = lc.Lightcone(shape, lc.HostBlocks(indptr, indices, data), scale)
    rows = [0, 5, 4 * 30 + 2, 4 * 62 + 3]
    a, b = cone.run_probes(rows, 5, workers=1), cone.run_probes(rows, 5, workers=2)
    assert np.array_equal(a[0], b[0])
    assert all(np.array_equal(x[2], y[2]) and np.array_equal(x[1], y[1]) for x, y in zip(a[1], b[1]))
