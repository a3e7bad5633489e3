"""Incremental updates (SURVEY 8f-3, second half): re-entering ``with`` for a few keys and asking for an observable again
must not rebuild the compacted matrix and the step kernels' copies of it -- and must give exactly what a rebuild gives.

The reference's scatter touches only the keys set (bodge/hamiltonian.py:102-118) and its parameter sweeps rely on it
(tests/test_physics.py:155-160, 221-224).  Here ``bdg_scatter`` patches the blocks it writes into the compacted BSR,
the fixed-width rows, the block dictionary (new blocks are appended) and the direction codes, and restricts the
Hermitian check to those blocks; a changed zero pattern, a full table or an off-site block that breaks the DFMA
kernels' precondition fall back to the rebuild.  ``bdg_stats`` tells which path ran.
"""

import numpy as np
import pytest

import cases
from oracle import bdg_oracle as orc
from util import rel_err, same_bits

pytestmark = pytest.mark.gpu
TOL = 1e-10


def _oracle_state(system_recorder_blocks, shape):
    indptr, indices = orc.cubic_skeleton(shape)
    data = orc.zero_data(indices)
    for packed in system_recorder_blocks:
        orc.scatter(indptr, indices, data, *packed)
    return orc.eliminate_zeros(indptr, indices, data)


def _check(system, blocks, shape, kernels, n_cols=8, n_moments=24):
    """Exported matrix == oracle over all with-blocks so far (bit for bit); moments of every kernel == oracle."""
    ptr, idx, dat = _oracle_state(blocks, shape)
    ex = system.matrix("bsr")
    assert np.array_equal(ex.indptr, ptr) and np.array_equal(ex.indices, idx)
    assert same_bits(ex.data, dat)
    H = orc.to_scipy(ptr, idx, dat)
    scale = 1.01 * orc.norm_inf(ptr, idx, dat)
    assert abs(system.spectral_bound() - scale) <= 1e-12 * scale
    want = orc.cheb_moments(H, orc.rademacher(4, H.shape[0], np.arange(n_cols)), n_moments, scale)
    out = {}
    for kernel in kernels:
        got = system.chebyshev_moments(n_moments, vectors=n_cols, seed=4, scale=scale, kernel=kernel)
        assert rel_err(got, want) <= TOL, kernel
        out[kernel] = got
    return out


def _fresh(gpu_api, shape, blocks):
    """The same final state assembled from scratch (one fill per with-block)."""
    system = gpu_api.Hamiltonian(gpu_api.CubicLattice(shape))
    for packed in blocks:
        system.fill(*packed)
    return system


def _onsite(sites, lattice, mats, pair=None):
    """Packed with-block: on-site H (and optionally Δ) for a list of sites."""
    i = np.array([lattice.index(s) for s in sites], dtype=np.int32)
    h = np.array(mats, dtype=np.complex128).reshape(-1, 2, 2)
    if pair is None:
        return (i, i, h, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 2, 2), np.complex128))
    return (i, i, h, i, i, np.array(pair, dtype=np.complex128).reshape(-1, 2, 2))


CASES = {
    # tag: (shape, packed builder, kernels that apply)
    "junction_24_18_1": ((24, 18, 1), "junction", ("auto", "pair", "t2", "dict_diag", "dict", "ell", "dmma")),
    "readme_3d_6_5_4": ((6, 5, 4), "swave_3d", ("auto", "t2", "dict_diag", "dict", "ell", "dmma")),
    "dwave_12_14_1": ((12, 14, 1), "dwave_rashba", ("auto", "pair", "t2", "dict", "ell", "dmma")),
    "disordered_16_20_1": ((16, 20, 1), "disordered_swave", ("auto", "pair", "t2", "dict_diag", "ell")),
}


@pytest.mark.parametrize("tag", sorted(CASES))
def test_patched_copies_equal_a_rebuild(gpu_api, tag):
    import bodge_b200 as b
    from bodge_b200 import workloads

    shape, build, kernels = CASES[tag]
    lattice = b.CubicLattice(shape)
    blocks = [getattr(workloads, build)(shape)]
    system = _fresh(gpu_api, shape, blocks)
    _check(system, blocks, shape, kernels)
    base = system._sys.stats()
    rng = np.random.default_rng(7)
    σ0, σ1, σ3, jσ2 = b.σ0, b.σ1, b.σ3, b.jσ2

    # (1) a handful of on-site terms get NEW values (new dictionary entries), zero pattern unchanged: patched in place
    sites = [tuple(int(v) for v in rng.integers(0, shape)) for _ in range(7)]
    sites = list(dict.fromkeys(sites))
    blocks.append(_onsite(sites, lattice, [(2.0 + 0.1 * k) * σ0 - 0.3 * σ3 for k in range(len(sites))]))
    system.fill(*blocks[-1])
    got = _check(system, blocks, shape, kernels)
    st = system._sys.stats()
    assert st["patched_scatters"] == base["patched_scatters"] + 1, st
    assert st["native_builds"] == base["native_builds"] and st["compactions"] == base["compactions"], st
    assert st["listed_hermitian_checks"] == base["listed_hermitian_checks"] + 1
    fresh = _fresh(gpu_api, shape, blocks)
    want = _check(fresh, blocks, shape, kernels)
    for kernel in kernels:  # same matrix, same arithmetic: the patched copies give bit-identical moments
        assert np.array_equal(got[kernel], want[kernel]), kernel

    # (2) a quarter of all sites get ONE common new on-site block and gap (the spin-valve sweep of the reference's tests;
    # an update that rewrites more than a quarter of all BLOCKS takes the rebuild path by design: step 6)
    half = [s for s in lattice.sites() if s[0] < max(1, shape[0] // 4)]
    blocks.append(_onsite(half, lattice, [3.0 * σ0 + 0.4 * σ3] * len(half), pair=[-0.25 * jσ2] * len(half)))
    system.fill(*blocks[-1])
    got = _check(system, blocks, shape, kernels)
    st2 = system._sys.stats()
    assert st2["patched_scatters"] == st["patched_scatters"] + 1 and st2["native_builds"] == st["native_builds"], st2
    want = _check(_fresh(gpu_api, shape, blocks), blocks, shape, kernels)
    for kernel in kernels:
        assert np.array_equal(got[kernel], want[kernel]), kernel

    # (3) writing the same values again changes nothing and stays on the fast path
    system.fill(*blocks[-1])
    blocks.append(blocks[-1])
    _check(system, blocks, shape, kernels)
    assert system._sys.stats()["native_builds"] == st["native_builds"]

    # (4) an on-site term set to ZERO changes the zero pattern: rebuild (and still right)
    blocks.append(_onsite([sites[0]], lattice, [0.0 * σ0], pair=[0.0 * jσ2]))
    system.fill(*blocks[-1])
    _check(system, blocks, shape, kernels)
    st4 = system._sys.stats()
    assert st4["native_builds"] == st["native_builds"] + 1 and st4["compactions"] == st["compactions"] + 1, st4

    # (5) an off-site block that is not real-diagonal: kernels that rely on real-diagonal hopping must let go of it
    i, j = (1, 1, 0) if shape[2] == 1 else (1, 1, 1), (2, 1, 0) if shape[2] == 1 else (2, 1, 1)
    hop = -1.0 * σ0 + 0.2j * σ1
    blocks.append((np.array([lattice.index(i), lattice.index(j)], np.int32), np.array([lattice.index(j), lattice.index(i)], np.int32),
                   np.array([hop, hop.conj().T]), np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 2, 2), np.complex128)))
    system.fill(*blocks[-1])
    # (on three-dimensional lattices the even-vector kernel needs real-diagonal hopping blocks as well)
    drop = ("dict_diag", "t2") if shape[1] > 1 and shape[2] > 1 else ("dict_diag",)
    _check(system, blocks, shape, [k for k in kernels if k not in drop])

    # (6) rewriting the whole Hamiltonian in one block: streaming rebuild instead of one warp per block
    before = system._sys.stats()
    system.fill(*blocks[0])
    blocks.append(blocks[0])
    _check(system, blocks, shape, [k for k in kernels if k not in drop])
    after = system._sys.stats()
    assert after["patched_scatters"] == before["patched_scatters"] and after["native_builds"] == before["native_builds"] + 1, after


def test_patch_past_the_cube_kernels_dictionary_limit(gpu_api):
    """The even-vector kernel for three-dimensional lattices holds at most 64 distinct blocks.  A patch that adds more
    keeps the copies, takes that kernel out of the plan, and the other kernels carry on with the patched dictionary."""
    import bodge_b200 as b
    from bodge_b200 import workloads

    shape = (6, 5, 4)
    lattice = b.CubicLattice(shape)
    blocks = [workloads.swave_3d(shape)]
    system = _fresh(gpu_api, shape, blocks)
    system.chebyshev_moments(16, vectors=2000, seed=1)
    assert system._sys.cheb_format()["kernel"] == "t2"
    base = system._sys.stats()

    sites = list(lattice.sites())[:70]  # 70 new on-site blocks, less than a quarter of all blocks: the patch path
    blocks.append(_onsite(sites, lattice, [(2.0 + 0.01 * k) * b.σ0 - 0.3 * b.σ3 for k in range(len(sites))]))
    system.fill(*blocks[-1])
    st = system._sys.stats()
    assert st["patched_scatters"] == base["patched_scatters"] + 1, st
    assert st["native_builds"] == base["native_builds"] and st["compactions"] == base["compactions"], st
    with pytest.raises(ValueError):
        system._sys.cheb_begin(n_random=8, seed=1, scale=10.0, kernel="t2")
    system.chebyshev_moments(16, vectors=2000, seed=1)
    assert system._sys.cheb_format()["kernel"] == "dict_diag" and system._sys.cheb_format()["distinct_blocks"] > 64
    _check(system, blocks, shape, ("auto", "dict_diag", "dict", "ell"))
    assert system._sys.stats()["native_builds"] == base["native_builds"]


def test_dict_api_sweep_stays_incremental(gpu_api):
    """The reference's idiom verbatim: a loop that re-enters `with` for some on-site terms and asks for the free energy
    (tests/test_physics.py:175-228).  One build, then patches only; values equal those of freshly built systems."""
    import bodge_b200 as b

    shape = (14, 9, 1)
    lattice = gpu_api.CubicLattice(shape)
    system = cases.readme_swave(gpu_api, shape)
    F = []
    for k, theta in enumerate(np.linspace(0.0, np.pi, 4)):
        with system as (H, D):
            for i in lattice.sites():
                if i[0] >= shape[0] // 2:
                    H[i, i] = 3.0 * gpu_api.σ0 - 0.3 * (np.cos(theta) * gpu_api.σ3 + np.sin(theta) * gpu_api.σ1)
        F.append(system.free_energy(0.1, cuda=True, scale=9.0))
        fresh = cases.readme_swave(gpu_api, shape)
        with fresh as (H, D):
            for i in lattice.sites():
                if i[0] >= shape[0] // 2:
                    H[i, i] = 3.0 * gpu_api.σ0 - 0.3 * (np.cos(theta) * gpu_api.σ3 + np.sin(theta) * gpu_api.σ1)
        assert F[-1] == fresh.free_energy(0.1, cuda=True, scale=9.0)
        assert abs(F[-1] - fresh.free_energy(0.1)) <= 1e-10 * abs(F[-1])   # ... and the reference's dense algorithm
    st = system._sys.stats()
    assert st["native_builds"] == 1 and st["patched_scatters"] == 3, st
    assert isinstance(b.__version__, str)


def test_failed_checks_leave_a_consistent_state(gpu_api):
    """A non-Hermitian update raises like the reference and leaves the matrix modified (hamiltonian.py:121-122); the
    copies follow the matrix, and the next update re-checks everything."""
    shape = (9, 8, 1)
    system = cases.readme_swave(gpu_api, shape)
    system.chebyshev_moments(8, vectors=8, seed=1)
    with pytest.raises(RuntimeError):
        with system as (H, D):
            H[(2, 2, 0), (2, 2, 0)] = 1j * gpu_api.σ1
    # the stored (non-Hermitian) matrix is what every export sees
    ex = system.matrix("bsr")
    k = system.index((2, 2, 0), (2, 2, 0))
    assert np.array_equal(system._matrix.data[k][:2, :2], 1j * gpu_api.σ1)
    assert ex.shape == system.shape
    # a Hermitian value restores it; the check after a failed one is a full one
    before = system._sys.stats()["listed_hermitian_checks"]
    with system as (H, D):
        H[(2, 2, 0), (2, 2, 0)] = 3.0 * gpu_api.σ0
    assert system._sys.stats()["listed_hermitian_checks"] == before
    Hs = system.matrix("bsr")
    scale = system.spectral_bound()
    want = orc.cheb_moments(Hs, orc.rademacher(1, Hs.shape[0], np.arange(8)), 16, scale)
    for kernel in ("auto", "pair", "dict_diag", "ell"):
        assert rel_err(system.chebyshev_moments(16, vectors=8, seed=1, scale=scale, kernel=kernel), want) <= TOL
    # pairs outside the skeleton still raise IndexError and leave the copies usable
    with pytest.raises(IndexError):
        with system as (H, D):
            H[(0, 0, 0), (5, 5, 0)] = gpu_api.σ0
    assert rel_err(system.chebyshev_moments(16, vectors=8, seed=1, scale=scale), want) <= TOL
