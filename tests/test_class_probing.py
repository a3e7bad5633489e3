"""CPU checks behind ``density_matrix`` / ``order_parameter`` / ``selfconsistent`` with ``spacing=``: the distance classes
of ``bodge_b200.probing`` against breadth-first distances on the lattice graph, and the class-sum prediction of
``class_oracle.py`` against the recursion on class columns.  The GPU twin is ``test_gpu_class_probing.py``."""

import itertools
import math
import os
import re

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import shortest_path

import class_oracle as co
import fermi_oracle as fo
from bodge_b200 import _native, kpm, probing, workloads
from oracle import bdg_oracle as orc
from util import oracle_assemble

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T = 0.1


def hop_distances(shape, wraps):
    """All-pairs hop counts on the nearest-neighbour graph of ``CubicLattice(shape)`` (flat index ``z + Lz(y + Ly x)``),
    with the face-to-face edges of the wrapping axes only."""
    idx = np.arange(int(np.prod(shape))).reshape(shape)
    i, j = [], []
    for axis in range(3):
        L = shape[axis]
        if L >= 2:
            i.append(np.take(idx, range(L - 1), axis=axis).ravel())
            j.append(np.take(idx, range(1, L), axis=axis).ravel())
        if wraps[axis] and L >= 3:
            i.append(np.take(idx, [L - 1], axis=axis).ravel())
            j.append(np.take(idx, [0], axis=axis).ravel())
    i, j = (np.concatenate(a) if a else np.zeros(0, int) for a in (i, j))
    n = idx.size
    graph = coo_matrix((np.ones(len(i)), (i, j)), shape=(n, n)).tocsr()
    return shortest_path(graph, directed=False, unweighted=True)


def rule_count(L, s, wraps):
    if not wraps:
        return min(L, s)
    return L if L < s else math.ceil(L / (L // s))


SHAPES = [(1, 1, 1), (2, 1, 1), (7, 1, 1), (6, 4, 1), (9, 6, 1), (13, 5, 1), (2, 7, 3), (5, 4, 3), (11, 2, 1)]


@pytest.mark.parametrize("shape", SHAPES)
def test_classes_keep_their_sites_apart(shape):
    for wraps in itertools.product((False, True), repeat=3):
        dist = hop_distances(shape, wraps)
        for s in (1, 2, 3, 4, 5, 6, 7, 9, 14):
            cls, n_classes = probing.site_classes(shape, s, wraps)
            assert cls.dtype == np.int32 and cls.shape == (int(np.prod(shape)),)
            assert n_classes == math.prod(rule_count(L, s, w) for L, w in zip(shape, wraps))
            assert set(np.unique(cls)) == set(range(n_classes))  # every class is used
            same = (cls[:, None] == cls[None, :]) & ~np.eye(len(cls), dtype=bool)
            if same.any():
                assert dist[same].min() >= s, (shape, wraps, s)


@pytest.mark.parametrize("L", [1, 2, 3, 5, 7, 16, 17, 31, 32, 33, 97, 1000, 1024])
def test_axis_class_counts(L):
    for s in (1, 2, 3, 5, 8, 16, 31, 32, 33):
        for wraps in (False, True):
            c = probing.axis_classes(L, s, wraps)
            assert c.min() == 0 and c.max() + 1 == rule_count(L, s, wraps)
            for a in range(L):  # the coordinates of one class are >= s apart, cyclically when the axis wraps
                other = np.flatnonzero(c == c[a])
                d = np.abs(other - a)
                d = np.minimum(d, L - d) if wraps else d
                assert np.all((d == 0) | (d >= s)), (L, s, wraps, a)


def test_uniform_tiling_of_a_divisible_torus():
    """1024 = 64 runs of 16: the classes of a wrapping axis are x mod 16, the same tiling as an open axis."""
    assert np.array_equal(probing.axis_classes(1024, 16, True), np.arange(1024) % 16)


def test_bad_arguments():
    for L, s in ((0, 2), (3, 0), (-1, 1)):
        with pytest.raises(ValueError):
            probing.axis_classes(L, s, False)


def assembled(build, shape):
    _, (ptr, idx, dat) = oracle_assemble(shape, [build(shape)])
    return orc.to_scipy(ptr, idx, dat), 1.01 * orc.norm_inf(ptr, idx, dat)


@pytest.mark.parametrize("name,shape,wraps", [
    ("readme", (6, 5, 1), (False, False, False)),
    ("periodic", (7, 5, 1), (True, True, False)),
    ("dwave_rashba", (5, 6, 1), (False, False, False)),
])
@pytest.mark.parametrize("spacing", [1, 2, 3])
def test_class_sum_prediction_is_the_class_recursion(name, shape, wraps, spacing):
    build = {"readme": workloads.readme_swave, "periodic": lambda s: workloads.junction(s, periodic=True),
             "dwave_rashba": workloads.dwave_rashba}[name]
    H, scale = assembled(build, shape)
    n_coef = kpm.free_energy_moments(T, scale)[0]
    cls, n_classes = probing.site_classes(shape, spacing, wraps)
    class_rows = (4 * np.arange(n_classes)[:, None] + np.arange(4)).ravel()
    n = int(np.prod(shape))
    Ly = shape[1]
    # on-site blocks of every site, and a few bonds (read at i from the columns of class(j))
    pairs = [(i, i) for i in range(n)] + [(7, 8), (8, 7), (7, 7 + Ly), (12, 12 - Ly)]
    i = np.array([p[0] for p in pairs])
    j = np.array([p[1] for p in pairs])
    read_col = (4 * cls[j][:, None] + np.arange(4)).ravel()
    read_site = np.repeat(i, 4)
    got = co.class_local_kpm(H, cls, class_rows, read_col, read_site, T, n_coef, scale)
    P = co.polynomial_dense(H, T, n_coef, scale)
    want = co.class_sum(P, cls, class_rows, read_col, read_site)
    assert np.max(np.abs(got - want)) <= 1e-12
    # the same polynomial read on unit columns is today's path; its own sites alone are the class sum with one member
    exact = fo.fermi_local_kpm(H, (4 * j[:, None] + np.arange(4)).ravel(), np.arange(4 * len(pairs)), read_site, T, n_coef,
                               scale)
    lone = cls[j][:, None] == cls[None, :]  # members of class(j)
    if lone.sum(axis=1).max() == 1:
        assert np.max(np.abs(got - exact)) <= 1e-12
    else:
        assert np.max(np.abs(got - exact)) > 1e-12  # the other members contribute


def test_wide_spacing_reads_the_exact_elements():
    """spacing >= n_coef: every other member of a class lies beyond the series' reach, so a class read is the exact read."""
    shape = (13, 4, 1)
    H, scale = assembled(workloads.readme_swave, shape)
    n_coef = 10  # degree 9; spacing 10 on a 13-long open axis leaves classes of two or one members
    cls, n_classes = probing.site_classes(shape, n_coef, (False, False, False))
    assert np.bincount(cls).max() == 2
    class_rows = 4 * np.arange(n_classes) + 3
    sites = np.arange(52)
    got = co.class_local_kpm(H, cls, class_rows, cls[sites], sites, T, n_coef, scale)
    exact = fo.fermi_local_kpm(H, 4 * sites + 3, sites, sites, T, n_coef, scale)
    assert np.max(np.abs(got - exact)) <= 1e-14


def test_new_abi_symbols():
    header = open(os.path.join(REPO, "include", "bdg.h")).read()
    for name, n_args in (("bdg_set_classes", 4), ("bdg_gather_blocks", 4)):
        assert re.search(rf"^int {name}\(", header, flags=re.M)
        assert len(_native.SIGNATURES[name]) == n_args
    assert re.search(r"BDG_X0_CLASS = 2", header) and _native.X0_CLASS == 2
    for method in ("set_classes", "gather_blocks"):
        assert callable(getattr(_native.System, method))
