"""``Hamiltonian.density_matrix`` / ``order_parameter`` / ``selfconsistent`` on the GPU: local elements of the Fermi
function read by the accumulator of the Chebyshev recursion, against the exact ``f(H)`` (``eigh``) and the dense
fixed point of the gap equation.  CPU twin: ``test_density_oracle.py``."""

import warnings

import numpy as np
import pytest

import cases
import fermi_oracle as fo
from bodge_b200 import workloads
from util import same_bits

pytestmark = pytest.mark.gpu
T = 0.1
TOL = 1e-10


def junction_periodic(api, shape):
    system = api.Hamiltonian(api.CubicLattice(shape))
    system.fill(*workloads.junction(shape, periodic=True))
    return system


SYSTEMS = {
    "open_2d": (lambda api: cases.readme_swave(api, (8, 7, 1)), [((3, 3, 0), (3, 4, 0)), ((0, 0, 0), (1, 0, 0))]),
    "periodic_2d": (lambda api: junction_periodic(api, (9, 6, 1)), [((0, 2, 0), (8, 2, 0)), ((4, 0, 0), (4, 5, 0))]),
    "cube_3d": (lambda api: cases.swave_3d(api, (4, 4, 3)), [((1, 2, 1), (1, 2, 2)), ((2, 1, 0), (3, 1, 0))]),
    "dwave_rashba": (lambda api: cases.dwave_rashba(api, (6, 7, 1)), [((2, 3, 0), (3, 3, 0)), ((2, 3, 0), (2, 2, 0))]),
    "junction_phase": (lambda api: cases.junction(api, (12, 5, 1)), [((3, 2, 0), (4, 2, 0)), ((8, 1, 0), (8, 2, 0))]),
}


def dense_blocks(system, rho, pairs):
    lat = system.lattice
    return np.stack([rho[4 * lat[i]:4 * lat[i] + 4, 4 * lat[j]:4 * lat[j] + 4] for i, j in pairs])


@pytest.fixture(scope="module")
def readme(gpu_api):
    system = cases.readme_swave(gpu_api, (8, 7, 1))
    return system, fo.fermi_dense(system.matrix("dense"), T)


@pytest.mark.parametrize("name", list(SYSTEMS))
def test_blocks_equal_dense_fermi(gpu_api, name):
    build, bonds = SYSTEMS[name]
    system = build(gpu_api)
    sites = [(1, 1, 0), (0, 0, 0), bonds[0][0]] if name != "cube_3d" else [(1, 1, 1), (0, 0, 0), (3, 3, 2)]
    pairs = [(s, s) for s in sites] + bonds + [(j, i) for i, j in bonds]
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        got = system.density_matrix(T, pairs)
    want = dense_blocks(system, fo.fermi_dense(system.matrix("dense"), T), pairs)
    assert got.shape == (len(pairs), 4, 4) and got.dtype == np.complex128
    assert np.max(np.abs(got - want)) <= TOL
    assert system._sys.cheb_format()["kernel"] != "t2"  # "auto" keeps every vector


def test_every_kernel_agrees(readme):
    system, rho = readme
    pairs = [((3, 3, 0), (3, 3, 0)), ((3, 3, 0), (3, 4, 0)), ((7, 6, 0), (6, 6, 0))]
    want = dense_blocks(system, rho, pairs)
    ref = system.density_matrix(T, pairs, kernel="pair")
    assert system._sys.cheb_format()["kernel"] == "pair"
    assert np.max(np.abs(ref - want)) <= TOL
    for kernel in ("dict_diag", "dict", "ell", "dmma"):
        got = system.density_matrix(T, pairs, kernel=kernel)
        assert system._sys.cheb_format()["kernel"] == kernel
        assert np.max(np.abs(got - ref)) <= 1e-12, kernel
    auto = system.density_matrix(T, pairs)
    assert system._sys.cheb_format()["kernel"] in ("pair", "dict_diag")
    assert np.max(np.abs(auto - ref)) <= 1e-12


def test_small_batches_give_the_same_blocks(readme):
    system, rho = readme
    pairs = [((x, y, 0), (x, (y + 1) % 7, 0)) for x in range(0, 8, 2) for y in range(0, 7, 3)]
    whole = system.density_matrix(T, pairs)
    batched = system.density_matrix(T, pairs, batch=8)
    assert np.max(np.abs(batched - whole)) <= 1e-13
    assert np.max(np.abs(whole - dense_blocks(system, rho, pairs))) <= TOL


def test_refusals(readme):
    system, _ = readme
    on_site = [((1, 1, 0), (1, 1, 0))]
    with pytest.raises(ValueError, match="even-vector"):
        system.density_matrix(T, on_site, kernel="t2")
    for bad_T in (0.0, -0.1):
        with pytest.raises(ValueError):
            system.density_matrix(bad_T, on_site)
        with pytest.raises(ValueError):
            system.order_parameter(bad_T, 1.0)
    with pytest.raises(IndexError):
        system.density_matrix(T, [((1, 1, 0), (3, 3, 0))])  # not a block of the skeleton
    with pytest.raises(ValueError):
        system.density_matrix(T, [((1, 1, 0), (8, 1, 0))])  # outside the 8 x 7 lattice
    with pytest.warns(Warning, match="truncate the Fermi series"):
        system.density_matrix(T, on_site, moments=64)


def test_zero_hamiltonian_gives_half_identity(gpu_api):
    system = gpu_api.Hamiltonian(gpu_api.CubicLattice((4, 3, 1)))
    got = system.density_matrix(T, [((1, 1, 0), (1, 1, 0)), ((1, 1, 0), (2, 1, 0))])
    assert np.array_equal(got[0], 0.5 * np.eye(4)) and not got[1].any()
    assert not system.order_parameter(T, 1.0).any()


def test_moments_unchanged_by_a_preceding_density_matrix(gpu_api):
    system = cases.dwave_rashba(gpu_api, (6, 7, 1))
    before = system.chebyshev_moments(64, vectors=8, seed=3)
    system.density_matrix(T, [((2, 3, 0), (3, 3, 0))])
    after = system.chebyshev_moments(64, vectors=8, seed=3)
    assert same_bits(before, after)


def test_order_parameter_equals_dense(gpu_api):
    system = cases.junction(gpu_api, (12, 5, 1))
    rho = fo.fermi_dense(system.matrix("dense"), T)
    lat = system.lattice
    sites = [(0, 0, 0), (5, 2, 0), (11, 4, 0)]
    want = np.array([-1.5 * rho[4 * lat[s], 4 * lat[s] + 3] for s in sites])
    assert np.max(np.abs(system.order_parameter(T, 1.5, sites) - want)) <= TOL
    potential = {(0, 0, 0): 1.5, (5, 2, 0): 0.0, (11, 4, 0): 2.5}
    got = system.order_parameter(T, potential)  # the V = 0 site is left out
    assert np.max(np.abs(got - want[[0, 2]] * np.array([1.0, 2.5 / 1.5]))) <= TOL
    d = 4 * np.arange(lat.size)
    full = system.order_parameter(T, 1.5)
    assert full.shape == (lat.size,) and np.max(np.abs(full + 1.5 * rho[d, d + 3])) <= TOL


@pytest.fixture(scope="module")
def converged(gpu_api):
    """The 6 x 6 open lattice (H[i,i] = σ0, bonds -σ0, V = 2, T = 0.05) iterated from Δ_i = 0.1."""
    L, V, T_ = 6, 2.0, 0.05
    lat = gpu_api.CubicLattice((L, L, 1))
    system = gpu_api.Hamiltonian(lat)
    with system as (H, D):
        for i in lat.sites():
            H[i, i] = 1.0 * gpu_api.σ0
            D[i, i] = 0.1 * gpu_api.jσ2
        for i, j in lat.bonds():
            H[i, j] = -1.0 * gpu_api.σ0
    delta, it = system.selfconsistent(T_, V, tol=1e-10)
    return system, delta, it, V, T_


def test_selfconsistent_reproduces_the_dense_fixed_point(converged):
    system, delta, it, V, T_ = converged
    want, _ = fo.gap_fixed_point(6, V, T_, tol=1e-12)
    assert np.max(np.abs(delta - want)) <= 1e-8
    assert abs(it - fo.gap_fixed_point(6, V, T_, tol=1e-10)[1]) <= 2
    d = 4 * np.arange(36)
    assert np.max(np.abs(np.asarray(system.matrix("dense"))[d, d + 3] - delta)) == 0  # the state stays in the system
    with pytest.warns(Warning, match="no convergence"):
        system.selfconsistent(T_, V, tol=0.0, max_iter=2)


def test_converged_gap_makes_the_free_energy_stationary(converged):
    system, delta, _, V, T_ = converged
    jσ2 = np.array([[0.0, 1.0], [-1.0, 0.0]])
    sites = np.arange(36)
    h = 1e-5

    def omega(d):
        system.fill((), (), (), sites, sites, d[:, None, None] * jσ2)
        return system.free_energy(T_, cuda=False) + np.sum(np.abs(d) ** 2) / V

    worst = 0.0
    for k in range(36):
        for unit in (1.0, 1j):
            dp, dm = delta.copy(), delta.copy()
            dp[k] += unit * h
            dm[k] -= unit * h
            worst = max(worst, abs(omega(dp) - omega(dm)) / (2 * h))
    system.fill((), (), (), sites, sites, delta[:, None, None] * jσ2)
    assert worst <= 1e-6
