"""``density_matrix`` / ``order_parameter`` / ``selfconsistent`` with ``spacing=``: Fermi reads from distance-classed start
columns (``bodge_b200.probing``, ``BDG_X0_CLASS``) against the CPU class-sum prediction of ``class_oracle.py`` and, when
the spacing is beyond the series' reach, against the one-column-per-site path.  CPU twin: ``test_class_probing.py``."""

import tracemalloc
import warnings

import numpy as np
import pytest

import cases
import class_oracle as co
from bodge_b200 import kpm, probing, workloads

pytestmark = pytest.mark.gpu
T = 0.1


def filled(api, shape, build):
    system = api.Hamiltonian(api.CubicLattice(shape))
    system.fill(*build(shape))
    return system


# name: (builder, wrapping axes, bond pairs)
SYSTEMS = {
    "open_2d": (lambda api: cases.readme_swave(api, (8, 7, 1)), (False, False, False),
                [((3, 3, 0), (3, 4, 0)), ((0, 0, 0), (1, 0, 0))]),
    "periodic_2d": (lambda api: filled(api, (9, 6, 1), lambda s: workloads.junction(s, periodic=True)), (True, True, False),
                    [((0, 2, 0), (8, 2, 0)), ((4, 0, 0), (4, 5, 0))]),
    "cube_3d": (lambda api: cases.swave_3d(api, (4, 4, 3)), (False, False, False),
                [((1, 2, 1), (1, 2, 2)), ((2, 1, 0), (3, 1, 0))]),
    "dwave_rashba": (lambda api: cases.dwave_rashba(api, (6, 7, 1)), (False, False, False),
                     [((2, 3, 0), (3, 3, 0)), ((2, 3, 0), (2, 2, 0))]),
    "junction_phase": (lambda api: cases.junction(api, (12, 5, 1)), (False, False, False),
                       [((3, 2, 0), (4, 2, 0)), ((8, 1, 0), (8, 2, 0))]),
    "disordered": (lambda api: filled(api, (7, 6, 1), workloads.disordered_swave), (False, False, False),
                   [((3, 3, 0), (4, 3, 0)), ((6, 5, 0), (6, 4, 0))]),
}


def class_reads(P, cls, pairs, lat):
    """Prediction for ``density_matrix(pairs, spacing)``: ``Σ_{j' in class(j)} P[4i:4i+4, 4j':4j'+4]``."""
    n_classes = int(cls.max()) + 1
    Q = P @ co.class_columns(P.shape[0], cls, np.arange(4 * n_classes))  # column 4k + β: class k, component β
    return np.stack([Q[4 * lat[i]:4 * lat[i] + 4, 4 * cls[lat[j]]:4 * cls[lat[j]] + 4] for i, j in pairs])


@pytest.mark.parametrize("name", list(SYSTEMS))
def test_reads_equal_the_class_sum_prediction(gpu_api, name):
    build, wraps, bonds = SYSTEMS[name]
    system = build(gpu_api)
    lat = system.lattice
    assert system._wrapping_axes() == wraps
    scale = system.spectral_bound()
    n_coef = kpm.free_energy_moments(T, scale)[0]
    P = co.polynomial_dense(np.asarray(system.matrix("dense")), T, n_coef, scale)
    pairs = [(s, s) for s in lat.sites()] + bonds + [(j, i) for i, j in bonds]
    d = 4 * np.arange(lat.size)
    for spacing in (1, 2, 5, n_coef):
        cls, _ = probing.site_classes(lat.shape, spacing, wraps)
        assert np.array_equal(system._classes(spacing), cls)
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            blocks = system.density_matrix(T, pairs, spacing=spacing)
            delta = system.order_parameter(T, 1.3, spacing=spacing)
        assert np.max(np.abs(blocks - class_reads(P, cls, pairs, lat))) <= 1e-12, spacing
        want = -1.3 * (P @ co.class_columns(P.shape[0], cls, 4 * np.arange(int(cls.max()) + 1) + 3))[d, cls]
        assert np.max(np.abs(delta - want)) <= 1e-12, spacing
        if spacing >= n_coef:
            assert np.max(np.abs(blocks - system.density_matrix(T, pairs))) <= 1e-12
            assert np.max(np.abs(delta - system.order_parameter(T, 1.3))) <= 1e-12
        assert system._sys.cheb_format()["kernel"] != "t2"


@pytest.fixture(scope="module")
def readme(gpu_api):
    return cases.readme_swave(gpu_api, (8, 7, 1))


def test_every_kernel_and_batching_agree(readme):
    system = readme
    pairs = [(s, s) for s in system.lattice.sites()] + [((3, 3, 0), (3, 4, 0)), ((7, 6, 0), (6, 6, 0))]
    ref = system.density_matrix(T, pairs, kernel="pair", spacing=2)
    assert system._sys.cheb_format()["kernel"] == "pair"
    for kernel in ("dict_diag", "dict", "ell", "dmma"):
        got = system.density_matrix(T, pairs, kernel=kernel, spacing=2)
        assert system._sys.cheb_format()["kernel"] == kernel
        assert np.max(np.abs(got - ref)) <= 1e-12, kernel
    whole = system.density_matrix(T, pairs, spacing=2)
    assert np.max(np.abs(whole - ref)) <= 1e-12
    for batch in (8, 6):  # 4 classes x 4 columns: 6 splits the four columns of a class over two batches
        assert np.max(np.abs(system.density_matrix(T, pairs, spacing=2, batch=batch) - whole)) <= 1e-13, batch
    op = system.order_parameter(T, 1.0, spacing=3)  # 9 columns: batches of 8 cut the class list
    assert np.max(np.abs(system.order_parameter(T, 1.0, spacing=3, batch=8) - op)) <= 1e-13


def test_refusals(gpu_api, readme):
    system = readme
    on_site = [((1, 1, 0), (1, 1, 0))]
    with pytest.raises(ValueError, match="even-vector"):
        system.density_matrix(T, on_site, kernel="t2", spacing=2)
    for bad in (0, -3, 1.5, True, "2"):
        with pytest.raises(ValueError, match="spacing"):
            system.density_matrix(T, on_site, spacing=bad)
        with pytest.raises(ValueError, match="spacing"):
            system.order_parameter(T, 1.0, spacing=bad)

    class Ring(gpu_api.CubicLattice.__mro__[1]):  # a Lattice that is no CubicLattice: six sites on a ring
        def index(self, coord):
            return coord[0]

        def sites(self):
            yield from ((x, 0, 0) for x in range(6))

        def bonds(self):
            for x in range(6):
                yield (x, 0, 0), ((x + 1) % 6, 0, 0)
                yield ((x + 1) % 6, 0, 0), (x, 0, 0)

        def edges(self):
            yield from ()

    ring = gpu_api.Hamiltonian(Ring((6, 1, 1)))
    with ring as (H, D):
        for i in ring.lattice.sites():
            H[i, i] = 0.5 * gpu_api.σ0
    with pytest.raises(ValueError, match="CubicLattice"):
        ring.density_matrix(T, [((0, 0, 0), (0, 0, 0))], spacing=2)
    with pytest.raises(ValueError, match="CubicLattice"):
        ring.selfconsistent(T, 1.0, spacing=2)


def test_start_vectors_are_the_class_indicators(gpu_api, readme):
    system = readme
    sysn = system._sys
    cls = system._classes(3)
    n_classes = int(cls.max()) + 1
    rows = np.array([4 * k + b for k in range(n_classes) for b in range(4)][::-1] + [7, 3])  # any order, repeats allowed
    for kernel in ("auto", "dmma"):
        sysn.cheb_begin(class_rows=rows, scale=system.spectral_bound(), kernel=kernel)
        t0 = sysn.cheb_vectors(len(rows), which=1)  # bdg_cheb_begin took the first step: T_{n-1} is T_0
        assert np.array_equal(t0, co.class_columns(4 * system.lattice.size, cls, rows))
    with pytest.raises(ValueError, match="column 1: class row"):
        sysn.cheb_begin(class_rows=[3, 4 * n_classes], scale=1.0)
    with pytest.raises(ValueError, match="column 0: class row -1"):
        sysn.cheb_begin(class_rows=[-1], scale=1.0)
    bad = cls.copy()
    bad[5] = n_classes
    with pytest.raises(ValueError, match="site 5: class"):
        sysn.set_classes(bad, n_classes)
    bad[5] = -1
    with pytest.raises(ValueError, match="site 5: class"):
        sysn.set_classes(bad, n_classes)
    with pytest.raises(ValueError, match="site classes given"):
        sysn.set_classes(cls[:-1], n_classes)
    with pytest.raises(ValueError, match="entry 1: block position"):
        sysn.gather_blocks([0, sysn.n_blocks])
    fresh = gpu_api.Hamiltonian(gpu_api.CubicLattice((3, 3, 1)))
    with pytest.raises(ValueError, match="no site classes"):
        fresh._sys.cheb_begin(class_rows=[3], scale=1.0)


def test_zero_hamiltonian_gives_the_class_sum_of_half_identity(gpu_api):
    system = gpu_api.Hamiltonian(gpu_api.CubicLattice((4, 3, 1)))
    pairs = [((1, 1, 0), (1, 1, 0)), ((1, 1, 0), (2, 1, 0)), ((1, 1, 0), (1, 2, 0))]
    one_class = system.density_matrix(T, pairs, spacing=1)  # f(H) = 1/2: every read's class holds the read site
    assert all(np.array_equal(b, 0.5 * np.eye(4)) for b in one_class)
    two = system.density_matrix(T, pairs, spacing=2)  # (1, 1) and (2, 1) differ in class, (1, 1) and (1, 2) too
    assert np.array_equal(two[0], 0.5 * np.eye(4)) and not two[1:].any()
    assert not system.order_parameter(T, 1.0, spacing=2).any()


def six_by_six(api):
    """The 6 x 6 open lattice of test_gpu_density.py (H[i,i] = σ0, bonds -σ0, start Δ_i = 0.1)."""
    lat = api.CubicLattice((6, 6, 1))
    system = api.Hamiltonian(lat)
    with system as (H, D):
        for i in lat.sites():
            H[i, i] = 1.0 * api.σ0
            D[i, i] = 0.1 * api.jσ2
        for i, j in lat.bonds():
            H[i, j] = -1.0 * api.σ0
    return system


def test_gap_equation(gpu_api):
    V, T_, tol = 2.0, 0.05, 1e-10
    exact, _ = six_by_six(gpu_api).selfconsistent(T_, V, tol=tol)
    wide_sys = six_by_six(gpu_api)
    n_coef = kpm.free_energy_moments(T_, wide_sys.spectral_bound())[0]
    wide, _ = wide_sys.selfconsistent(T_, V, tol=tol, spacing=n_coef)
    assert np.max(np.abs(wide - exact)) <= 1e-10
    small_sys = six_by_six(gpu_api)
    small, it = small_sys.selfconsistent(T_, V, tol=tol, spacing=3)
    assert it < 500
    again = small_sys.order_parameter(T_, V, spacing=3)  # the fixed point of the probed map
    assert np.max(np.abs(again - small)) <= tol
    assert np.max(np.abs(small - exact)) > tol  # ... which is not the exact one at this spacing


def uniform_torus(api, L):
    """README model on an L x L torus: its periodic edges filled with the bond value -σ0."""
    system = api.Hamiltonian(api.CubicLattice((L, L, 1)))
    h_i, h_j, h_val, p_i, p_j, p_val = workloads.readme_swave((L, L, 1))
    for axis in (0, 1):
        lo, hi = system.lattice.edges_array(axis)
        h_i = np.concatenate([h_i, lo, hi])
        h_j = np.concatenate([h_j, hi, lo])
        h_val = np.concatenate([h_val, np.broadcast_to(-api.σ0, (2 * len(lo), 2, 2))])
    system.fill(h_i, h_j, h_val, p_i, p_j, p_val)
    return system


def test_every_site_of_a_million_site_torus(gpu_api):
    moments = 200  # degree 199 < 256: neither torus below wraps around within the series' reach
    big = uniform_torus(gpu_api, 1024)
    assert big._wrapping_axes() == (True, True, False)
    N = big.lattice.size
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # moments below what tol asks for
        big.order_parameter(T, 1.0, sites=[(0, 0, 0)], spacing=16, moments=moments)  # classes uploaded, buffers sized
        tracemalloc.start()
        delta = big.order_parameter(T, 1.0, spacing=16, moments=moments)
        _, peak = tracemalloc.get_traced_memory()
        tracemalloc.stop()
        del big
        small = uniform_torus(gpu_api, 512).order_parameter(T, 1.0, spacing=16, moments=moments)
    assert delta.shape == (N,)
    assert np.max(np.abs(delta - delta[0])) <= 1e-12  # the class tiling of 1024 = 64 x 16 is uniform
    assert np.max(np.abs(small - delta[0])) <= 1e-12
    assert abs(delta[0]) > 1e-3
    assert peak <= 256 * N, f"{peak / N:.0f} bytes per site"  # one [N, 4] complex array and O(N) indices, any batch count
