"""Parity of the CUDA Chebyshev/KPM engine with the oracle (scipy bsr_matvecs recursion on the
same matrix) and, through free_energy / ldos, with the reference's own observables.

Tolerances (BASELINE.json north_star): moments and free energy within 1e-10 relative.
Moments are compared norm-wise (max|Δμ| / max|μ|): high orders pass through zero (SURVEY H6).
"""

import numpy as np
import pytest

import cases
from oracle import bdg_oracle as orc
from util import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-10


def scipy_of(system):
    return system.matrix("bsr")


@pytest.fixture(scope="module")
def random_system(gpu_api):
    return cases.random_periodic(gpu_api, (3, 5, 7), seed=11)


@pytest.mark.parametrize("kernel", ["ell", "dmma", "fma"])
@pytest.mark.parametrize("n_cols", [1, 2, 3, 4, 5, 8, 12, 19])
def test_random_column_moments(random_system, kernel, n_cols):
    system = random_system
    H = scipy_of(system)
    scale = system.spectral_bound()
    x0 = orc.rademacher(99, H.shape[0], np.arange(n_cols))
    want = orc.cheb_moments(H, x0, 64, scale)
    got = system.chebyshev_moments(64, vectors=n_cols, seed=99, scale=scale, kernel=kernel)
    assert got.shape == want.shape
    assert rel_err(got, want) <= TOL
    summed = system.chebyshev_moments(64, vectors=n_cols, seed=99, scale=scale, kernel=kernel, summed=True)
    assert rel_err(summed, want.sum(axis=1)) <= TOL


@pytest.mark.parametrize("kernel", ["ell", "dmma", "fma"])
def test_probe_moments_match_fixture(gpu_api, observables, kernel):
    """Fixture = scipy recursion on the REFERENCE's own matrix("bsr")."""
    builders = {"readme_12_12_1": lambda: cases.readme_swave(gpu_api, (12, 12, 1)),
                "random_3_5_7": lambda: cases.random_periodic(gpu_api, (3, 5, 7), seed=11),
                "dwave_9_8_1": lambda: cases.dwave_rashba(gpu_api, (9, 8, 1))}
    for tag, make in builders.items():
        system = make()
        want = observables[f"mu_{tag}"]
        scale, site = float(observables[f"mu_{tag}_scale"]), int(observables[f"mu_{tag}_site"])
        assert abs(system.spectral_bound() - scale) <= 1e-12 * scale
        probes = system.chebyshev_moments(want.shape[0], rows=[4 * site + a for a in range(4)], scale=scale, kernel=kernel)
        random = system.chebyshev_moments(want.shape[0], vectors=4, seed=1234, scale=scale, kernel=kernel)
        assert rel_err(probes, want[:, :4]) <= TOL
        assert rel_err(random, want[:, 4:]) <= TOL


@pytest.mark.parametrize("kernel", ["ell", "dmma", "fma"])
def test_recursion_vectors(random_system, kernel):
    """The vectors themselves after a few steps: T_n and T_{n-1} against the scipy recursion."""
    system = random_system
    H = scipy_of(system)
    scale = system.spectral_bound()
    n_cols, steps = 5, 6
    x0 = orc.rademacher(5, H.shape[0], np.arange(n_cols) + 3)
    t_prev, t_cur = x0, (H / scale) @ x0
    for _ in range(steps):
        t_prev, t_cur = t_cur, orc.cheb_step(H / scale, t_cur, t_prev)
    sysn = system._sys
    sysn.cheb_begin(n_random=n_cols, seed=5, col_offset=3, scale=scale, kernel=kernel)
    sysn.cheb_steps(steps)
    assert np.max(np.abs(sysn.cheb_vectors(n_cols, 0) - t_cur)) <= 1e-12 * np.max(np.abs(t_cur))
    assert np.max(np.abs(sysn.cheb_vectors(n_cols, 1) - t_prev)) <= 1e-12 * np.max(np.abs(t_prev))
    sysn.cheb_end()


def test_start_vectors_are_the_oracles(random_system):
    sysn = random_system._sys
    n_rows = random_system.shape[0]
    sysn.cheb_begin(n_random=11, seed=42, col_offset=7, scale=50.0)
    assert np.array_equal(sysn.cheb_vectors(11, 1), orc.rademacher(42, n_rows, np.arange(11) + 7))
    rows = [0, 5, n_rows - 1, 17, 17]
    sysn.cheb_begin(probe_rows=rows, scale=50.0)
    assert np.array_equal(sysn.cheb_vectors(5, 1), orc.probes(n_rows, rows))
    sysn.cheb_end()


def test_moment_properties_and_determinism(random_system):
    system = random_system
    rows = np.arange(0, system.shape[0], 13)
    a = system.chebyshev_moments(200, rows=rows)
    b = system.chebyshev_moments(200, rows=rows)
    assert np.array_equal(a, b)                       # fixed-order reductions: bitwise repeatable
    assert np.array_equal(a[0], np.ones(len(rows)))   # <e|e> = 1
    assert np.max(np.abs(a)) <= 1 + 1e-12             # |<x|T_n|x>| <= <x|x>
    fma = system.chebyshev_moments(200, rows=rows, kernel="fma")
    assert rel_err(fma, a) <= 1e-12
    # batching the columns must not change anything
    c = system.chebyshev_moments(200, rows=rows, batch=8)
    assert np.array_equal(a, c)
    # odd number of moments
    d = system.chebyshev_moments(7, rows=rows[:3])
    assert np.array_equal(d, a[:7, :3])


@pytest.mark.parametrize("tag", ["snf_10_7_3", "readme_12_12_1", "junction_30_10_1", "dwave_9_8_1"])
def test_free_energy_matches_reference(gpu_api, observables, tag):
    """free_energy(T, cuda=True) (KPM, exact trace) vs the reference's dense eigvalsh values."""
    from test_oracle import SMALL

    system = SMALL[tag](gpu_api)
    for T, F_ref in zip(observables["temps"], observables[f"F_{tag}"]):
        if T >= 0.05:
            F = system.free_energy(float(T), cuda=True)
            assert abs(F - F_ref) <= TOL * abs(F_ref), (tag, T, F, F_ref)
        elif T > 0:
            F = system.free_energy(float(T), cuda=True, moments=4096)
            assert abs(F - F_ref) <= 1e-6 * abs(F_ref)
    F0 = system.free_energy(0.0, cuda=True, moments=2048)
    assert abs(F0 - observables[f"F_{tag}"][0]) <= 1e-4 * abs(F0)   # kink at ε=0: algebraic convergence
    # the reference's own CPU-vs-GPU test template (tests/test_hamiltonian.py:421-425)
    for T in [0.1, 1.0]:
        assert np.allclose(system.free_energy(T, cuda=False), system.free_energy(T, cuda=True))
    with pytest.raises(Exception):
        system.free_energy(-1.0, cuda=True)


def test_free_energy_C1_exact_trace(gpu_api, observables):
    """Config C1 (40x40): all 6400 unit columns, vs the reference's dense value at T = 0.1."""
    system = cases.readme_swave(gpu_api, (40, 40, 1))
    temps, F_ref = observables["temps"], observables["F_C1"]
    F01 = system.free_energy(0.1, cuda=True)
    assert abs(F01 - F_ref[list(temps).index(0.1)]) <= TOL * abs(F01)
    F10 = system.free_energy(1.0, cuda=True)
    assert abs(F10 - F_ref[list(temps).index(1.0)]) <= TOL * abs(F10)
    # stochastic trace: unbiased estimate, error ~ 1/sqrt(R * 4N)
    Fs = system.free_energy(0.1, cuda=True, vectors=64, seed=1234)
    assert abs(Fs - F01) <= 1e-2 * abs(F01)


@pytest.mark.parametrize("tag,site", [("readme_12_12_1", (6, 6, 0)), ("random_5_5_2", (2, 3, 1)), ("dwave_9_8_1", (4, 4, 0))])
def test_ldos_matches_reference(gpu_api, observables, tag, site):
    from test_oracle import SMALL

    system = SMALL[tag](gpu_api)
    got = system.ldos(site, observables["ldos_E"])
    assert rel_err(got, observables[f"ldos_{tag}"]) <= TOL
    got = system.ldos(site, list(observables["ldos_E"]), kernel="fma")
    assert rel_err(got, observables[f"ldos_{tag}"]) <= TOL


def test_ldos_positive_everywhere(gpu_api):
    # reference tests/test_hamiltonian.py:467-500
    system = cases.random_periodic(gpu_api, (5, 5, 2), seed=21)
    sites = [(i, j, k) for i in range(5) for j in range(5) for k in range(2)]
    rho = system.ldos_map(sites, [0.0, 0.01, 0.10, 0.50, 1.00, 2.00, 4.00])
    assert rho.shape == (50, 7) and (rho >= 0).all()


def test_magnetic_isotropy(gpu_api):
    """Rotating a homogeneous exchange field changes neither F nor the LDOS (rtol 1e-10), the
    reference's tests/test_physics.py:115-172 on the KPM path."""
    api = gpu_api
    lattice = api.CubicLattice((128, 1, 1))
    system = api.Hamiltonian(lattice)
    with system as (H, D):
        for i in lattice.sites():
            D[i, i] = -0.1 * api.jσ2
        for i, j in lattice.bonds():
            H[i, j] = -1.0 * api.σ0
    T, i0, E0 = 0.05, (64, 0, 0), [0.0, 0.05]
    F0 = system.free_energy(T, cuda=True, scale=2.4)
    r0 = system.ldos(i0, E0, scale=2.4)[0]
    rng = np.random.default_rng(4)
    Fs, rs = [], []
    for _ in range(4):
        th, ph = 2 * np.pi * rng.random(2)
        s = np.cos(th) * api.σ1 + np.sin(th) * np.cos(ph) * api.σ2 + np.sin(th) * np.sin(ph) * api.σ3
        with system as (H, D):
            for i in lattice.sites():
                H[i, i] = -0.05 * s
        Fs.append(system.free_energy(T, cuda=True, scale=2.4))
        rs.append(system.ldos(i0, E0, scale=2.4)[0])
    assert all(not np.allclose(F0, F, rtol=1e-10) for F in Fs)
    assert all(not np.allclose(r0, r, rtol=1e-10) for r in rs)
    assert all(np.allclose(a, b, rtol=1e-10) for a, b in zip(Fs[:-1], Fs[1:]))
    assert all(np.allclose(a, b, rtol=1e-9) for a, b in zip(rs[:-1], rs[1:]))


def test_full_size_chebyshev_properties(gpu_api):
    """C5 (10^6 sites, k = 8): properties that hold independent of size."""
    import bodge_b200 as b
    from bodge_b200 import workloads

    shape = (1000, 1000, 1)
    system = b.Hamiltonian(b.CubicLattice(shape))
    system.fill(*workloads.junction(shape))
    mu = system.chebyshev_moments(32, vectors=8, seed=1234)
    assert np.array_equal(mu[0], np.full(8, 4e6))            # <x|x> = 4N exactly for +-1 vectors
    assert np.max(np.abs(mu)) <= 4e6 * (1 + 1e-12)
    assert np.max(np.abs(mu[1::2])) < 4e6 * 0.01              # odd moments ~ Tr-odd ~ 0 (± spectrum)
    fma = system.chebyshev_moments(32, vectors=8, seed=1234, kernel="fma")
    assert rel_err(fma, mu) <= 1e-12
    # column sharding: columns 4..7 computed alone (as another GPU would) are bit-identical
    sysn = system._sys
    sysn.cheb_begin(n_random=4, seed=1234, col_offset=4, scale=system.spectral_bound())
    sysn.cheb_steps(15)
    part = sysn.cheb_read(32, 4)
    assert rel_err(part, mu[:, 4:]) <= 1e-13
    # a small twin of the same model agrees with the oracle end to end
    small = b.Hamiltonian(b.CubicLattice((30, 10, 1)))
    small.fill(*workloads.junction((30, 10, 1)))
    H = small.matrix("bsr")
    want = orc.cheb_moments(H, orc.rademacher(1234, H.shape[0], np.arange(8)), 32, small.spectral_bound())
    assert rel_err(small.chebyshev_moments(32, vectors=8, seed=1234), want) <= TOL


# ---- the fixed-width (ELL) step kernel: format edge cases ------------------------------------
def _moments_vs_oracle(system, n_cols, kernel, n_moments=48, seed=7):
    H = scipy_of(system)
    scale = system.spectral_bound()
    want = orc.cheb_moments(H, orc.rademacher(seed, H.shape[0], np.arange(n_cols)), n_moments, scale)
    got = system.chebyshev_moments(n_moments, vectors=n_cols, seed=seed, scale=scale, kernel=kernel)
    return rel_err(got, want)


def test_ell_rows_without_diagonal_block(gpu_api):
    """Pure hopping model: no H[i,i], no Δ[i,i] -> eliminate_zeros drops every diagonal block and
    slot 0 of every ELL row is padding; T_n[row] must still be found."""
    lattice = gpu_api.CubicLattice((6, 5, 1))
    system = gpu_api.Hamiltonian(lattice)
    with system as (H, D):
        for i, j in lattice.bonds():
            H[i, j] = -1.0 * gpu_api.σ0 + 0.3j * (j[0] - i[0] + j[1] - i[1]) * gpu_api.σ3
            if i[0] < 3:
                D[i, j] = 0.2 * gpu_api.jσ2
                D[j, i] = 0.2 * gpu_api.jσ2
    ex = system.matrix("bsr")
    assert not any(r in ex.indices[ex.indptr[r] : ex.indptr[r + 1]] for r in range(lattice.size))
    for kernel in ("ell", "dmma"):
        assert _moments_vs_oracle(system, 5, kernel) <= TOL
    # mixed: some rows with, some without a diagonal block
    with system as (H, D):
        for i in lattice.sites():
            if (i[0] + i[1]) % 3 == 0:
                H[i, i] = 0.7 * gpu_api.σ0 + 0.1 * gpu_api.σ1
    assert _moments_vs_oracle(system, 9, "ell") <= TOL


@pytest.mark.parametrize("n_cols", [16, 17, 24, 33, 40, 70])
def test_ell_many_columns_share_one_matrix_pass(random_system, n_cols):
    """k > 8: panels are processed in groups of up to four per pass over the matrix, the last
    group ragged (n_panels = 2, 3, 3, 5, 5, 9)."""
    assert _moments_vs_oracle(random_system, n_cols, "ell") <= TOL
    a = random_system.chebyshev_moments(20, vectors=n_cols, seed=3, kernel="ell")
    b = random_system.chebyshev_moments(20, vectors=n_cols, seed=3, kernel="dmma")
    assert rel_err(a, b) <= 1e-12
    # per-column results do not depend on which panel/group a column lands in
    c = random_system.chebyshev_moments(20, vectors=n_cols, seed=3, kernel="ell", batch=8)
    assert rel_err(c, a) <= 1e-13


@pytest.mark.parametrize("shape", [(1, 1, 1), (5, 1, 1), (2, 2, 2), (4, 4, 1), (3, 3, 3)])
def test_ell_row_widths(gpu_api, shape):
    """Row widths 1 (padded to 3), 3, 4, 5 and 7."""
    system = cases.random_periodic(gpu_api, shape, seed=5)
    assert _moments_vs_oracle(system, 3, "ell") <= TOL
    assert _moments_vs_oracle(system, 11, "ell") <= TOL


def test_long_rows_fall_back_to_the_generic_kernel(gpu_api):
    """A lattice whose rows exceed 8 blocks cannot use the fixed-width format: auto picks the
    BSR kernel, and asking for kernel='ell' explicitly is an error."""
    import bodge_b200 as b

    class Dense1D(b.CubicLattice):
        """Chain with bonds to the 1st..5th neighbours (11 blocks per interior row)."""

        def bonds(self, axis=None):
            for x in range(self.shape[0]):
                for d in range(1, 6):
                    if x + d < self.shape[0]:
                        yield (x, 0, 0), (x + d, 0, 0)
                        yield (x + d, 0, 0), (x, 0, 0)

    lattice = Dense1D((40, 1, 1))
    system = b.Hamiltonian(lattice)
    with system as (H, D):
        for i in lattice.sites():
            H[i, i] = 0.3 * b.σ0
            D[i, i] = 0.1 * b.jσ2
        for i, j in lattice.bonds():
            H[i, j] = -(1.0 / abs(j[0] - i[0])) * b.σ0
    assert _moments_vs_oracle(system, 6, "auto") <= TOL
    with pytest.raises(ValueError):
        system.chebyshev_moments(8, vectors=2, kernel="ell")


# ---- observables evaluated on the device (csrc/observables.cu) -------------------------------
def test_device_resolvent_and_contraction(random_system):
    from bodge_b200 import kpm

    system = random_system
    n_mom, k = 300, 11
    scale = system.spectral_bound()
    mu = system.chebyshev_moments(n_mom, vectors=k, seed=21, scale=scale)
    sysn = system._sys
    sysn.cheb_begin(n_random=k, seed=21, scale=scale)
    sysn.cheb_steps(n_mom // 2 - 1)
    # resolvent diagonal at a few complex energies, both half planes
    z = np.array([0.1 + 0.05j, -0.4 + 0.02j, 0.0 + 0.1j, 0.7 - 0.03j])
    w, pref = kpm.resolvent_weights(z)
    got = sysn.kpm_resolvent(n_mom, k, w, pref)
    want = np.array([[kpm.resolvent_diagonal(mu[:, c], zz) for zz in z] for c in range(k)])
    assert got.shape == (k, len(z))
    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))
    # series contraction
    coef = np.cos(0.37 * np.arange(n_mom)) / (1 + np.arange(n_mom))
    per_col = sysn.kpm_contract(coef, k)
    assert np.allclose(per_col, coef @ mu, rtol=1e-12, atol=1e-12)
    total = sysn.kpm_contract(coef, k, summed=True)
    assert abs(total - float(coef @ mu.sum(axis=1))) <= 1e-12 * abs(total)
    # fewer moments than available, odd count
    per_col = sysn.kpm_contract(coef[:77], k)
    assert np.allclose(per_col, coef[:77] @ mu[:77], rtol=1e-12, atol=1e-12)
    sysn.cheb_end()


def test_ldos_map_many_sites_matches_single_site_calls(gpu_api):
    system = cases.dwave_rashba(gpu_api, (9, 8, 1))
    sites = [(x, y, 0) for x in range(0, 9, 2) for y in range(0, 8, 3)]
    E = np.linspace(-0.4, 0.4, 9)
    many = system.ldos_map(sites, E, moments=600)
    assert many.shape == (len(sites), len(E))
    for s in (0, 7, len(sites) - 1):
        one = system.ldos(sites[s], E, moments=600)
        assert np.allclose(many[s], one, rtol=1e-12, atol=1e-14)
    assert (many >= 0).all()


def test_full_size_ldos_map_C3(gpu_api):
    """C3 (100x100 d-wave + Rashba): LDOS at the 1024 probe sites of SURVEY 8d (4096 probe
    columns in one batch), size-independent checks only."""
    import bodge_b200 as b
    from bodge_b200 import workloads

    shape = (100, 100, 1)
    system = b.Hamiltonian(b.CubicLattice(shape))
    system.fill(*workloads.dwave_rashba(shape))
    sites = [(3 * p + 2, 3 * q + 2, 0) for p in range(32) for q in range(32)]
    E = np.linspace(-0.15, 0.15, 11)
    rho = system.ldos_map(sites, E, moments=768)
    assert rho.shape == (1024, 11) and np.isfinite(rho).all() and (rho >= 0).all()
    # a probe's result does not depend on which other columns share its batch / panel
    pick = [0, 517, 1023]
    alone = system.ldos_map([sites[i] for i in pick], E, moments=768)
    assert np.allclose(rho[pick], alone, rtol=1e-11, atol=1e-14)
    # bulk sites related by the lattice's C4 symmetry about the centre see the same LDOS ... up to
    # the finite-size asymmetry of the probe grid; the d-wave gap suppresses the LDOS at ε = 0
    bulk = rho[[i for i, s in enumerate(sites) if 30 <= s[0] < 70 and 30 <= s[1] < 70]]
    assert bulk[:, 5].mean() < 0.8 * bulk[:, 0].mean()


# ---- block-dictionary matrix format (kernel="dict") ---------------------------------------------
def _disordered(api, shape, seed=5):
    """Uniform hopping, site-dependent on-site potential and gap: every diagonal block distinct."""
    lattice = api.CubicLattice(shape)
    system = api.Hamiltonian(lattice)
    rng = np.random.default_rng(seed)
    with system as (H, D):
        for i in lattice.sites():
            H[i, i] = rng.normal() * api.σ0 + 0.3 * rng.normal() * api.σ3
            D[i, i] = -0.1 * rng.random() * api.jσ2
        for i, j in lattice.bonds():
            H[i, j] = -1.0 * api.σ0
    return system


DICT_SYSTEMS = {
    "readme_12_12_1": lambda api: cases.readme_swave(api, (12, 12, 1)),
    "junction_30_10_1": lambda api: cases.junction(api, (30, 10, 1)),
    "dwave_9_8_1": lambda api: cases.dwave_rashba(api, (9, 8, 1)),
    "swave3d_6_5_4": lambda api: cases.swave_3d(api, (6, 5, 4)),
    "chain_17_1_1": lambda api: cases.readme_swave(api, (17, 1, 1)),
    "disordered_11_9_1": lambda api: _disordered(api, (11, 9, 1)),
}


@pytest.mark.parametrize("tag", sorted(DICT_SYSTEMS))
def test_dictionary_format_is_bit_identical_to_ell(gpu_api, tag):
    """Same arithmetic in the same order on a de-duplicated copy of the blocks: not 1e-10, equal."""
    system = DICT_SYSTEMS[tag](gpu_api)
    H = scipy_of(system)
    scale = system.spectral_bound()
    for n_cols in (1, 3, 8, 19):
        ell = system.chebyshev_moments(48, vectors=n_cols, seed=3, scale=scale, kernel="ell")
        dic = system.chebyshev_moments(48, vectors=n_cols, seed=3, scale=scale, kernel="dict")
        assert np.array_equal(ell, dic)
        want = orc.cheb_moments(H, orc.rademacher(3, H.shape[0], np.arange(n_cols)), 48, scale)
        assert rel_err(dic, want) <= TOL
    sysn = system._sys
    sysn.cheb_begin(n_random=4, seed=1, scale=scale, kernel="auto")
    fmt = sysn.cheb_format()
    # few distinct blocks -> a dictionary format is the default; with real diagonal hopping blocks
    # (everything here but the d-wave + Rashba model) the DFMA variant of it
    offsite_diagonal = tag != "dwave_9_8_1"
    # (... on the small 2-D lattices among them, two steps per launch on an 8-column panel: test_gpu_pair.py; the d-wave model
    # too: its on-site blocks are real-diagonal, which makes the MMA rows light enough for the two-step kernel to pay)
    two_step = tag in ("readme_12_12_1", "junction_30_10_1", "disordered_11_9_1", "dwave_9_8_1")
    assert fmt["kernel"] == ("pair" if two_step else "dict_diag" if offsite_diagonal else "dict")
    if offsite_diagonal:
        for n_cols in (1, 4, 8, 19):
            got = system.chebyshev_moments(48, vectors=n_cols, seed=3, scale=scale, kernel="dict_diag")
            ref = system.chebyshev_moments(48, vectors=n_cols, seed=3, scale=scale, kernel="ell")
            assert rel_err(got, ref) <= 1e-13   # same sums, different rounding order
    else:
        with pytest.raises(ValueError):
            sysn.cheb_begin(n_random=4, seed=1, scale=scale, kernel="dict_diag")
        sysn.cheb_begin(n_random=4, seed=1, scale=scale, kernel="auto")
    n_slots_bytes = 260 * sysn.cheb_info()["n_blocks"]
    assert fmt["matrix_bytes_per_step"] < n_slots_bytes
    blocks = {blk.tobytes() for blk in H.data}
    # distinct stored blocks (+ the zero block used for padding slots / absent diagonals)
    assert len(blocks) <= fmt["distinct_blocks"] <= len(blocks) + 1
    sysn.cheb_end()


def test_dictionary_format_declines_matrices_without_repetition(random_system):
    sysn = random_system._sys
    scale = random_system.spectral_bound()
    sysn.cheb_begin(n_random=4, seed=1, scale=scale, kernel="auto")
    fmt = sysn.cheb_format()
    # the dictionary build gives up as soon as the distinct blocks exceed 35 % of all slots
    assert fmt["kernel"] == "ell" and fmt["distinct_blocks"] >= 0.35 * sysn.cheb_info()["n_blocks"]
    with pytest.raises(ValueError):
        sysn.cheb_begin(n_random=4, seed=1, scale=scale, kernel="dict")
    sysn.cheb_end()


def test_unassigned_kernel_numbers_are_refused(random_system):
    """4 and 5 name no kernel (include/bdg.h): bdg_cheb_begin refuses them like the numbers outside the enum."""
    from bodge_b200 import _native

    lib, sysn = _native.load(), random_system._sys
    for kernel in (4, 5, -1, 11):
        rc = lib.bdg_cheb_begin(sysn._h, _native.X0_RADEMACHER, 4, None, 1, 0, 10.0, kernel)
        assert rc == _native.E_INVALID and f"unknown kernel {kernel}" in _native.last_error()


def test_dictionary_format_with_every_block_distinct(gpu_api, monkeypatch):
    """Forced on a random matrix (table as large as the matrix): still exact."""
    monkeypatch.setenv("BDG_DICT_MAX_PERCENT", "100")
    system = cases.random_periodic(gpu_api, (3, 5, 7), seed=11)
    H = scipy_of(system)
    scale = system.spectral_bound()
    want = orc.cheb_moments(H, orc.rademacher(99, H.shape[0], np.arange(11)), 64, scale)
    got = system.chebyshev_moments(64, vectors=11, seed=99, scale=scale, kernel="dict")
    assert rel_err(got, want) <= TOL
    assert np.array_equal(got, system.chebyshev_moments(64, vectors=11, seed=99, scale=scale, kernel="ell"))


def test_dictionary_follows_matrix_updates(gpu_api):
    """A later `with` block changes blocks: the dictionary must be rebuilt, not reused."""
    system = cases.readme_swave(gpu_api, (10, 6, 1))
    scale = 9.0
    before = system.chebyshev_moments(32, vectors=4, seed=2, scale=scale, kernel="dict")
    with system as (H, D):
        H[(3, 2, 0), (3, 2, 0)] = 1.7 * gpu_api.σ0 + 0.2 * gpu_api.σ3
    after = system.chebyshev_moments(32, vectors=4, seed=2, scale=scale, kernel="dict")
    want = orc.cheb_moments(scipy_of(system), orc.rademacher(2, system.shape[0], np.arange(4)), 32, scale)
    assert not np.array_equal(before, after)
    assert rel_err(after, want) <= TOL


# ---- spectral bound from the recursion itself (SURVEY 8f-4) ---------------------------------------
@pytest.mark.parametrize("tag", ["dwave_9_8_1", "readme_12_12_1", "random_3_5_7", "junction_30_10_1", "swave3d_5_4_6"])
def test_lanczos_spectral_bound_is_safe_and_tighter(gpu_api, tag):
    from test_oracle import SMALL

    system = SMALL[tag](gpu_api)
    lam = float(np.max(np.abs(np.linalg.eigvalsh(np.asarray(system.matrix("dense"))))))
    loose = system.spectral_bound()
    tight = system.spectral_bound("lanczos")
    assert lam < tight <= loose
    assert tight <= 1.06 * lam
    # the tighter scale is usable: same free energy as with the row-sum bound, fewer moments needed
    F_loose = system.free_energy(0.1, cuda=True)
    F_tight = system.free_energy(0.1, cuda=True, scale=tight)
    assert abs(F_tight - F_loose) <= 1e-10 * abs(F_loose)
    with pytest.raises(ValueError):
        system.spectral_bound("power")


def test_boundedness_check_rejects_a_scale_that_is_too_small(gpu_api):
    """The acceptance test inside spectral_bound("lanczos"): at a scale below max|ε| the recursion blows up."""
    system = cases.readme_swave(gpu_api, (12, 12, 1))
    lam = float(np.max(np.abs(np.linalg.eigvalsh(np.asarray(system.matrix("dense"))))))
    ok = system.chebyshev_moments(258, vectors=4, seed=1, scale=1.001 * lam)[0::2]
    bad = system.chebyshev_moments(258, vectors=4, seed=1, scale=0.99 * lam)[0::2]
    assert np.all(ok <= ok[0] * (1 + 1e-9))
    assert not np.all(bad <= bad[0] * (1 + 1e-9))


# ---- BASELINE.json's full sizes: size-independent properties --------------------------------------
@pytest.mark.parametrize("cfg", ["C5", "C4"])
def test_full_size_recursion_properties(cfg):
    """10^6-site junction (C5) and 64^3 s-wave (C4), 8 stochastic columns: the matrix formats of the
    step kernel agree (the dictionary kernel's VECTORS are bit-identical to the plain copy's; its dot
    products are summed over a different partition of the rows -- the grid differs -- so moments agree
    to rounding; the DFMA variant to 1e-12), runs are bit-reproducible, mu_0 = <x|x> = 4N exactly,
    |mu_n| <= mu_0, and the recursion is linear: the summed moments equal the sum of the per-column moments."""
    import bodge_b200 as b
    from bodge_b200 import workloads

    c = workloads.CONFIGS[cfg]
    system = b.Hamiltonian(b.CubicLattice(c["shape"]))
    assert system.fill(*c["build"](c["shape"])) == 0.0
    n_rows = system.shape[0]
    scale = system.spectral_bound()
    runs = {k: system.chebyshev_moments(24, vectors=8, seed=1234, scale=scale, kernel=k) for k in ("ell", "dict", "dict_diag", "auto")}
    # auto (moments only): the even-vector recursion, two applications of H per pass -- cheb_pair.cu on the 2-D junction,
    # cheb_cube.cu (4-column panels) on the 3-D lattice
    assert system._sys.cheb_format()["kernel"] == "t2"
    assert system._sys.cheb_info()["panel_width"] == (8 if cfg == "C5" else 4)
    assert rel_err(runs["dict"], runs["ell"]) <= 1e-13
    assert rel_err(runs["auto"], runs["dict_diag"]) <= 1e-12
    if cfg == "C4":  # 134 MB per vector set: compare T_n itself after a few steps
        vecs = {}
        for k in ("ell", "dict"):
            system._sys.cheb_begin(n_random=8, seed=1234, scale=scale, kernel=k)
            system._sys.cheb_steps(5)
            vecs[k] = system._sys.cheb_vectors(8, 0)
        assert np.array_equal(vecs["dict"], vecs["ell"])
        del vecs
    assert rel_err(runs["dict_diag"], runs["ell"]) <= 1e-12
    mu = runs["auto"]
    assert np.array_equal(mu[0], np.full(8, float(n_rows)))
    assert np.all(np.abs(mu) <= n_rows * (1 + 1e-12))
    assert np.array_equal(mu, system.chebyshev_moments(24, vectors=8, seed=1234, scale=scale))
    summed = system.chebyshev_moments(24, vectors=8, seed=1234, scale=scale, summed=True)
    assert rel_err(summed, mu.sum(axis=1)) <= 1e-13
    # mu_1 = <x|H|x>/a for Rademacher x: Tr H = 0 for a BdG matrix, so mu_1 is pure sampling noise ~ sqrt(N)
    assert np.all(np.abs(mu[1]) < 50 * np.sqrt(n_rows))
    # generic-BSR kernel on the same matrix (no fixed-width copy, no dictionary)
    assert rel_err(system.chebyshev_moments(24, vectors=8, seed=1234, scale=scale, kernel="dmma"), runs["ell"]) <= 1e-12
