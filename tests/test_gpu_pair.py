"""The two-steps-per-pass Chebyshev kernel (kernel="pair", csrc/cheb_pair.cu; SURVEY 8f-4 temporal
blocking): T_{n+1} and T_{n+2} in one launch, T_{n+1} consumed out of shared memory.

Its row arithmetic is that of the single-step dictionary kernels, so the VECTORS must be bit-identical
to theirs for every patch / segment decomposition (halo values are recomputed, never exchanged); the
dot products are summed over another partition of the rows and agree to rounding; against the oracle
(scipy bsr_matvecs recursion) the moments hold the 1e-10 of BASELINE.json.
"""

import numpy as np
import pytest

import cases
from oracle import bdg_oracle as orc
from util import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-10

def _periodic(api, shape, *, x=True, y=True, random_hop=False, seed=3, disorder=False, onsite_pairing=True):
    """README-type s-wave system on a 2-D lattice with the reference's periodic edges filled in
    (bodge/lattice.py:161-197; tests/test_hamiltonian.py:17-57 fills them with random matrices): wrap-around
    bonds along x and / or the in-plane axis.  ``random_hop``: one of three random complex 2x2 matrices per bond
    (``H[j,i] = H[i,j]^†``), else ``-t σ0`` (real-diagonal blocks: the DFMA variant).  ``disorder``: random on-site
    potential and gap, so that every on-site block is distinct (the SELF path of the kernel)."""
    rng = np.random.default_rng(seed)
    lattice = api.CubicLattice(shape)
    system = api.Hamiltonian(lattice)
    in_plane = 1 if shape[2] == 1 else 2

    pool = [-1.0 * api.σ0 + 0.3 * (rng.random((2, 2)) - 0.5 + 1j * (rng.random((2, 2)) - 0.5)) for _ in range(3)]

    def hop():  # a few distinct complex matrices, so that the block dictionary still applies
        return pool[int(rng.integers(3))] if random_hop else -1.0 * api.σ0

    with system as (H, D):
        for i in lattice.sites():
            mu, ds = (3.0 + 0.4 * rng.random(), 0.1 + 0.2 * rng.random()) if disorder else (3.0, 0.2)
            H[i, i] = mu * api.σ0 - 0.05 * api.σ3
            if onsite_pairing:   # without it the on-site blocks are real-diagonal: two multiplications instead of two MMAs (SD)
                D[i, i] = -ds * api.jσ2
        pairs = list(lattice.bonds())
        if x:
            pairs += list(lattice.edges(axis=0))
        if y:
            pairs += list(lattice.edges(axis=in_plane))
        done = set()
        for i, j in pairs:
            if (i, j) in done:
                continue
            h = hop()
            H[i, j] = h
            H[j, i] = h.conj().T
            done.add((i, j))
            done.add((j, i))
    return system


SYSTEMS = {
    # tag: (builder, hopping blocks real-diagonal -> the pair kernel runs its DFMA variant)
    "readme_24_16_1": (lambda api: cases.readme_swave(api, (24, 16, 1)), True),
    "junction_30_40_1": (lambda api: cases.junction(api, (30, 40, 1)), True),      # two patches at P = 30
    "junction_9_1_67": (lambda api: cases.junction(api, (9, 1, 67)), True),        # planes along z, three patches
    "dwave_13_35_1": (lambda api: cases.dwave_rashba(api, (13, 35, 1)), False),    # complex hopping + bond pairing: DMMA rows
    "readme_3_3_1": (lambda api: cases.readme_swave(api, (3, 3, 1)), True),        # smallest lattice it accepts
    # the reference's PERIODIC skeleton with the edges filled in: the halo of the rim patches / segments is the opposite face
    "torus_11_17_1": (lambda api: _periodic(api, (11, 17, 1)), True),
    "torus_x_only_9_31_1": (lambda api: _periodic(api, (9, 31, 1), y=False), True),
    "torus_y_only_5_1_23": (lambda api: _periodic(api, (5, 1, 23), x=False), True),
    "torus_3_3_1": (lambda api: _periodic(api, (3, 3, 1)), True),                  # every site neighbours every plane
    "torus_random_hop_7_19_1": (lambda api: _periodic(api, (7, 19, 1), random_hop=True), False),
    "torus_disordered_10_16_1": (lambda api: _periodic(api, (10, 16, 1), disorder=True), True),   # > 64 distinct blocks: SELF path
    "open_disordered_12_33_1": (lambda api: _periodic(api, (12, 33, 1), x=False, y=False, disorder=True, random_hop=True), False),
    # general hopping blocks, real-diagonal on-site blocks (SD): held fragments / streamed per row (> 64 distinct blocks)
    "torus_normal_random_hop_8_17_1": (lambda api: _periodic(api, (8, 17, 1), random_hop=True, onsite_pairing=False), False),
    "open_normal_disordered_11_20_1": (lambda api: _periodic(api, (11, 20, 1), x=False, y=False, disorder=True, random_hop=True,
                                                             onsite_pairing=False), False),
}

# (BDG_PAIR_SEG, BDG_PAIR_P): None = planner's choice
PLANS = [(None, None), (5, 7), (1, 1), (4, 30), (3, 14), (1000, 2), (6, 22), (2, 5)]


def _set_plan(monkeypatch, plan):
    for name, value in zip(("BDG_PAIR_SEG", "BDG_PAIR_P"), plan):
        if value is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, str(value))


def _vectors(sysn, kernel, n_cols, steps, scale):
    sysn.cheb_begin(n_random=n_cols, seed=5, col_offset=3, scale=scale, kernel=kernel)
    sysn.cheb_steps(steps)
    out = sysn.cheb_vectors(n_cols, 0), sysn.cheb_vectors(n_cols, 1)
    fmt = sysn.cheb_format()["kernel"]
    sysn.cheb_end()
    return out, fmt


@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("tag", sorted(SYSTEMS))
def test_pair_vectors_are_bit_identical_to_the_single_step_kernel(gpu_api, monkeypatch, tag, plan):
    build, diag = SYSTEMS[tag]
    system = build(gpu_api)
    scale = system.spectral_bound()
    base = "dict_diag" if diag else "dict"
    _set_plan(monkeypatch, plan)
    # odd counts end on a single step; 1 = no pair at all; < 5 columns: padded to an 8-column panel (small lattices)
    for n_cols, steps in ((8, 6), (5, 7), (19, 2), (12, 1), (4, 6), (1, 5)):
        (cur, prev), fmt = _vectors(system._sys, "pair", n_cols, steps, scale)
        assert fmt == "pair"
        (want_cur, want_prev), fmt = _vectors(system._sys, base, n_cols, steps, scale)
        assert fmt == base
        if tag.startswith("torus"):
            # wrap-around neighbours: the single-step kernel adds a row's blocks in ascending block column, this one in
            # stencil direction (x-1, y-1, y+1, x+1) -- the same terms in another order where a neighbour wraps
            bound = 1e-13 * max(np.max(np.abs(want_cur)), 1.0)
            assert np.max(np.abs(cur - want_cur)) <= bound and np.max(np.abs(prev - want_prev)) <= bound
            continue
        assert np.array_equal(cur, want_cur), f"T_n differs: max {np.max(np.abs(cur - want_cur)):.3e}"
        assert np.array_equal(prev, want_prev), f"T_n-1 differs: max {np.max(np.abs(prev - want_prev)):.3e}"


@pytest.mark.parametrize("tag", sorted(SYSTEMS))
def test_pair_moments_match_the_oracle(gpu_api, monkeypatch, tag):
    build, diag = SYSTEMS[tag]
    system = build(gpu_api)
    H = system.matrix("bsr")
    scale = system.spectral_bound()
    for plan in PLANS[:3]:
        _set_plan(monkeypatch, plan)
        for n_cols, n_moments in ((8, 48), (5, 47), (19, 50), (12, 4), (8, 2), (4, 33), (2, 20)):
            got = system.chebyshev_moments(n_moments, vectors=n_cols, seed=3, scale=scale, kernel="pair")
            want = orc.cheb_moments(H, orc.rademacher(3, H.shape[0], np.arange(n_cols)), n_moments, scale)
            assert got.shape == want.shape
            assert rel_err(got, want) <= TOL
            single = system.chebyshev_moments(n_moments, vectors=n_cols, seed=3, scale=scale, kernel="dict_diag" if diag else "dict")
            assert rel_err(got, single) <= 1e-13   # same vectors, dot products summed in another order
            again = system.chebyshev_moments(n_moments, vectors=n_cols, seed=3, scale=scale, kernel="pair")
            assert np.array_equal(got, again)      # fixed-order reduction: bit-reproducible
    summed = system.chebyshev_moments(48, vectors=8, seed=3, scale=scale, kernel="pair", summed=True)
    assert rel_err(summed, system.chebyshev_moments(48, vectors=8, seed=3, scale=scale, kernel="pair").sum(axis=1)) <= 1e-13


def test_pair_probe_columns_and_ldos(gpu_api):
    """Unit start vectors (LDOS-type): sparse vectors spread one site per step, so halo handling errors
    show up as exact zeros / non-zeros in the wrong place."""
    system = cases.junction(gpu_api, (30, 40, 1))
    H = system.matrix("bsr")
    scale = system.spectral_bound()
    rows = [4 * system.lattice.index((x, y, 0)) + a for (x, y) in ((0, 0), (29, 39), (14, 29), (15, 30)) for a in (0, 3)]
    got = system.chebyshev_moments(64, rows=rows, scale=scale, kernel="pair")
    x0 = np.zeros((H.shape[0], len(rows)), dtype=np.complex128)
    x0[rows, np.arange(len(rows))] = 1.0
    assert rel_err(got, orc.cheb_moments(H, x0, 64, scale)) <= TOL
    E = np.linspace(-0.3, 0.3, 9)
    sites = [(14, 29, 0), (0, 39, 0)]   # 2 sites x 4 components = one 8-column panel
    assert rel_err(system.ldos_map(sites, E, kernel="pair"), system.ldos_map(sites, E, kernel="dict_diag")) <= 1e-12


def test_pair_declines_what_it_cannot_do(gpu_api):
    scale = 10.0
    three_d = cases.swave_3d(gpu_api, (6, 5, 4))._sys            # two-dimensional x-planes
    with pytest.raises(ValueError):
        three_d.cheb_begin(n_random=8, seed=1, scale=scale, kernel="pair")
    periodic = cases.random_periodic(gpu_api, (3, 5, 7), seed=11)._sys   # no dictionary, wrap-around bonds
    with pytest.raises(ValueError):
        periodic.cheb_begin(n_random=8, seed=1, scale=scale, kernel="pair")
    import bodge_b200 as b
    from bodge_b200 import workloads

    big = b.Hamiltonian(b.CubicLattice((260, 260, 1)))           # 67,600 sites: past the L2-resident size up to which
    big.fill(*workloads.readme_swave((260, 260, 1)))             # narrow column sets are padded to an 8-column panel
    with pytest.raises(ValueError):
        big._sys.cheb_begin(n_random=4, seed=1, scale=scale, kernel="pair")
    big._sys.cheb_begin(n_random=4, seed=1, scale=scale, kernel="auto")
    assert big._sys.cheb_format()["kernel"] == "dict_diag"
    big._sys.cheb_begin(n_random=5, seed=1, scale=scale, kernel="auto")
    assert big._sys.cheb_format()["kernel"] == "pair"
    del big
    flat = cases.readme_swave(gpu_api, (12, 12, 1))
    # wrap-around hopping along y: the torus geometry takes it (round 1 declined it)
    lattice = flat.lattice
    with flat as (H, D):
        for x in range(12):
            H[(x, 0, 0), (x, 11, 0)] = -1.0 * gpu_api.σ0
            H[(x, 11, 0), (x, 0, 0)] = -1.0 * gpu_api.σ0
    H2 = flat.matrix("bsr")
    want = orc.cheb_moments(H2, orc.rademacher(2, H2.shape[0], np.arange(8)), 16, flat.spectral_bound())
    for kernel in ("pair", "t2", "auto"):
        got = flat.chebyshev_moments(16, vectors=8, seed=2, kernel=kernel)
        assert flat._sys.cheb_format()["kernel"] == ("t2" if kernel == "auto" else kernel)
        assert rel_err(got, want) <= TOL
    assert lattice.size == 144
    short = cases.readme_swave(gpu_api, (2, 9, 1))              # fewer than 3 planes: x-1 and x+1 would be the same site
    with pytest.raises(ValueError):
        short._sys.cheb_begin(n_random=8, seed=1, scale=scale, kernel="pair")


def test_auto_prefers_pair_where_it_is_faster(gpu_api, monkeypatch):
    """kernel="auto": two steps per pass when the hopping blocks are real-diagonal (DFMA rows) and a panel has 8
    columns (or the lattice is small enough that narrow column sets are padded); single-step kernels otherwise;
    BDG_AUTO_PAIR=0 switches the preference off."""
    scale = 10.0
    flat = cases.readme_swave(gpu_api, (12, 12, 1))._sys
    for n_cols, want in ((8, "pair"), (19, "pair"), (5, "pair"), (4, "pair"), (1, "pair")):   # (small lattice: padded panels)
        flat.cheb_begin(n_random=n_cols, seed=1, scale=scale, kernel="auto")
        assert flat.cheb_format()["kernel"] == want
    monkeypatch.setenv("BDG_AUTO_PAIR", "0")
    flat.cheb_begin(n_random=8, seed=1, scale=scale, kernel="auto")
    assert flat.cheb_format()["kernel"] == "dict_diag"
    monkeypatch.delenv("BDG_AUTO_PAIR")
    dwave = cases.dwave_rashba(gpu_api, (9, 8, 1))._sys          # complex hopping blocks (MMA rows), real-diagonal on-site blocks (SD)
    dwave.cheb_begin(n_random=8, seed=1, scale=scale, kernel="auto")
    assert dwave.cheb_format()["kernel"] == "pair"
    pwave = _periodic(gpu_api, (9, 8, 1), x=False, y=False, random_hop=True)._sys   # complex hopping AND on-site pairing: ten MMAs per row
    pwave.cheb_begin(n_random=8, seed=1, scale=scale, kernel="auto")
    assert pwave.cheb_format()["kernel"] == "pair"
    monkeypatch.setenv("BDG_AUTO_PAIR", "0")
    pwave.cheb_begin(n_random=8, seed=1, scale=scale, kernel="auto")
    assert pwave.cheb_format()["kernel"] == "dict"
    monkeypatch.delenv("BDG_AUTO_PAIR")
    pwave.cheb_end()
    cube = cases.swave_3d(gpu_api, (6, 5, 4))._sys
    cube.cheb_begin(n_random=8, seed=1, scale=scale, kernel="auto")
    assert cube.cheb_format()["kernel"] == "dict_diag"
    for sysn in (flat, dwave, cube):
        sysn.cheb_end()


def test_pair_follows_matrix_updates(gpu_api):
    system = cases.readme_swave(gpu_api, (10, 12, 1))
    scale = system.spectral_bound() * 1.2
    before = system.chebyshev_moments(32, vectors=8, seed=2, scale=scale, kernel="pair")
    with system as (H, D):
        H[(4, 4, 0), (4, 4, 0)] = 0.7 * gpu_api.σ0 + 0.2 * gpu_api.σ3
    after = system.chebyshev_moments(32, vectors=8, seed=2, scale=scale, kernel="pair")
    assert not np.array_equal(before, after)
    Hm = system.matrix("bsr")
    assert rel_err(after, orc.cheb_moments(Hm, orc.rademacher(2, Hm.shape[0], np.arange(8)), 32, scale)) <= TOL


def test_one_call_c_entry_point(gpu_api):
    """bdg_cheb_moments -- begin + steps + read in one ABI call (SURVEY 8b) -- only returns moments, so it runs the
    even-vector recursion where that applies; checked at every moment count mod 4, per column and summed."""
    import ctypes as C

    from bodge_b200 import _native

    lib = _native.load()
    for system, want_kernel in ((cases.junction(gpu_api, (30, 40, 1)), "t2"), (cases.swave_3d(gpu_api, (6, 5, 4)), "dict_diag"),
                                (cases.dwave_rashba(gpu_api, (9, 8, 1)), "t2")):
        H = system.matrix("bsr")
        scale = system.spectral_bound()
        x0 = orc.rademacher(77, H.shape[0], np.arange(8) + 2)
        for n_moments in (1, 2, 3, 4, 5, 41, 42, 43, 44):
            want = orc.cheb_moments(H, x0, n_moments, scale)
            out = np.empty((n_moments, 8))
            _native.check(lib.bdg_cheb_moments(system._sys._h, _native.X0_RADEMACHER, 8, None, 77, 2, C.c_double(scale),
                                               n_moments, _native.MU_PER_COLUMN, out.ctypes.data_as(C.c_void_p), 0))
            assert rel_err(out, want) <= TOL
            total = np.empty(n_moments)
            _native.check(lib.bdg_cheb_moments(system._sys._h, _native.X0_RADEMACHER, 8, None, 77, 2, C.c_double(scale),
                                               n_moments, _native.MU_SUM, total.ctypes.data_as(C.c_void_p), 0))
            assert rel_err(total, want.sum(axis=1)) <= TOL
        assert system._sys.cheb_format()["kernel"] == want_kernel


def test_two_step_kernels_on_random_shapes_and_plans(monkeypatch):
    """Seeded sweep over lattice extents (either plane orientation), patch sizes, segment lengths, CTA shapes, column
    and step counts: pair vectors bit-identical to the single-step kernel, t2 vectors and moments to rounding."""
    import bodge_b200 as b
    from bodge_b200 import workloads

    rng = np.random.default_rng(2024)
    for case in range(24):
        Lx, M = int(rng.integers(3, 70)), int(rng.integers(3, 90))
        shape = (Lx, M, 1) if case % 3 else (Lx, 1, M)
        build = workloads.junction if case % 2 else workloads.readme_swave
        system = b.Hamiltonian(b.CubicLattice(shape))
        assert system.fill(*build(shape)) == 0.0
        scale = system.spectral_bound()
        plan = (int(rng.integers(1, Lx + 3)) if rng.random() < 0.7 else None,
                int(rng.integers(1, 31)) if rng.random() < 0.7 else None)
        _set_plan(monkeypatch, plan)
        n_cols, steps = int(rng.integers(1, 20)), int(rng.integers(1, 12))
        (cur, prev), fmt = _vectors(system._sys, "pair", n_cols, steps, scale)
        (want_cur, want_prev), _ = _vectors(system._sys, "dict_diag", n_cols, steps, scale)
        assert fmt == "pair", (shape, plan)
        assert np.array_equal(cur, want_cur) and np.array_equal(prev, want_prev), (shape, plan, n_cols, steps)
        n_mom = 2 * steps + int(rng.integers(0, 3))
        ref = system.chebyshev_moments(n_mom, vectors=n_cols, seed=9, scale=scale, kernel="dict_diag")
        for kernel in ("pair", "t2"):
            got = system.chebyshev_moments(n_mom, vectors=n_cols, seed=9, scale=scale, kernel=kernel)
            assert rel_err(got, ref) <= 1e-12, (shape, plan, n_cols, n_mom, kernel)
        sysn = system._sys
        sysn.cheb_begin(n_random=n_cols, seed=5, col_offset=3, scale=scale, kernel="t2")
        sysn.cheb_steps(2 * (steps // 2))                       # T_{2 (steps // 2) + 2}
        t2_cur = sysn.cheb_vectors(n_cols, 0)
        (want, _), _ = _vectors(sysn, "dict_diag", n_cols, 2 * (steps // 2) + 1, scale)
        assert np.max(np.abs(t2_cur - want)) <= 1e-13 * max(np.max(np.abs(want)), 1.0), (shape, plan)


# ---- the even-vector recursion (kernel="t2"): same kernel, E_{j+1} = 2 T_2(H~) E_j - E_{j-1} -------------------
@pytest.mark.parametrize("tag", sorted(SYSTEMS))
def test_t2_moments_match_the_oracle(gpu_api, monkeypatch, tag):
    """Three vector passes per two steps: only T_2j are kept, the four dot products of a launch give the same four
    moments (odd ones through a two-term recurrence).  Another rounding sequence than the three-term recursion,
    so: 1e-10 against the oracle (BASELINE.json), 1e-12 against the pair kernel, bit-reproducible."""
    build, diag = SYSTEMS[tag]
    system = build(gpu_api)
    H = system.matrix("bsr")
    scale = system.spectral_bound()
    for plan in PLANS[:4]:
        _set_plan(monkeypatch, plan)
        for n_cols, n_moments in ((8, 48), (5, 47), (19, 50), (12, 4), (8, 2), (8, 5), (6, 1), (8, 301), (4, 33), (1, 20), (3, 7)):
            got = system.chebyshev_moments(n_moments, vectors=n_cols, seed=3, scale=scale, kernel="t2")
            assert system._sys.cheb_format()["kernel"] == "t2"
            want = orc.cheb_moments(H, orc.rademacher(3, H.shape[0], np.arange(n_cols)), n_moments, scale)
            assert got.shape == want.shape
            assert rel_err(got, want) <= TOL
            pair = system.chebyshev_moments(n_moments, vectors=n_cols, seed=3, scale=scale, kernel="pair")
            assert rel_err(got, pair) <= 1e-12
            assert np.array_equal(got, system.chebyshev_moments(n_moments, vectors=n_cols, seed=3, scale=scale, kernel="t2"))
    summed = system.chebyshev_moments(48, vectors=8, seed=3, scale=scale, kernel="t2", summed=True)
    assert rel_err(summed, system.chebyshev_moments(48, vectors=8, seed=3, scale=scale, kernel="t2").sum(axis=1)) <= 1e-13


def test_t2_long_recursion_stays_within_tolerance(gpu_api):
    """4096 moments (2047 steps): the odd moments of the even-vector recursion come from a two-term recurrence along
    the launches, whose rounding error grows like sqrt(j) eps mu_0 -- far inside the 1e-10 of BASELINE.json."""
    system = cases.readme_swave(gpu_api, (24, 16, 1))
    H = system.matrix("bsr")
    scale = system.spectral_bound()
    got = system.chebyshev_moments(4096, vectors=8, seed=11, scale=scale, kernel="t2")
    want = orc.cheb_moments(H, orc.rademacher(11, H.shape[0], np.arange(8)), 4096, scale)
    assert rel_err(got, want) <= 1e-11
    assert rel_err(got, system.chebyshev_moments(4096, vectors=8, seed=11, scale=scale, kernel="pair")) <= 1e-11
    # ... and the observable built on them: exact-trace free energy against the dense spectrum
    F = system.free_energy(0.1, cuda=True)
    assert system._sys.cheb_format()["kernel"] == "t2"
    assert abs(F - system.free_energy(0.1)) <= 1e-10 * abs(F)


def test_t2_vectors_steps_and_incremental_reads(gpu_api):
    """bdg_cheb_begin takes the first step (T_2), bdg_cheb_steps advances in twos, T_n agrees with the three-term
    recursion to rounding, T_{n-1} is not kept; moments can be read between calls (the dot rows are brought
    into the single-step format incrementally)."""
    system = cases.junction(gpu_api, (30, 40, 1))
    sysn = system._sys
    scale = system.spectral_bound()
    sysn.cheb_begin(n_random=8, seed=5, col_offset=3, scale=scale, kernel="t2")
    assert sysn.cheb_available() == 4
    first = sysn.cheb_read(4, 8)
    sysn.cheb_steps(6)                       # three launches: T_8
    assert sysn.cheb_available() == 16
    mid = sysn.cheb_read(16, 8)
    sysn.cheb_steps(3)                       # rounded up to four steps: T_12
    assert sysn.cheb_available() == 24
    last = sysn.cheb_read(24, 8)
    t12 = sysn.cheb_vectors(8, 0)
    with pytest.raises(ValueError):
        sysn.cheb_vectors(8, 1)
    sysn.cheb_begin(n_random=8, seed=5, col_offset=3, scale=scale, kernel="dict_diag")
    sysn.cheb_steps(11)                      # T_12 by the three-term recursion
    want = sysn.cheb_vectors(8, 0)
    ref = sysn.cheb_read(24, 8)
    sysn.cheb_end()
    assert np.max(np.abs(t12 - want)) <= 1e-13 * np.max(np.abs(want))
    assert rel_err(last, ref) <= 1e-12
    assert np.array_equal(first, last[:4]) and np.array_equal(mid, last[:16])


def test_t2_observables_and_auto_moments(gpu_api):
    """chebyshev_moments / ldos_map / free_energy only read moments: their kernel="auto" is the even-vector
    recursion wherever kernel="auto" of the stepping API is the pair kernel."""
    system = cases.junction(gpu_api, (30, 40, 1))
    H = system.matrix("bsr")
    scale = system.spectral_bound()
    rows = [4 * system.lattice.index((x, y, 0)) + a for (x, y) in ((0, 0), (29, 39), (14, 29), (15, 30)) for a in (0, 3)]
    got = system.chebyshev_moments(64, rows=rows, scale=scale)
    assert system._sys.cheb_format()["kernel"] == "t2"
    x0 = np.zeros((H.shape[0], len(rows)), dtype=np.complex128)
    x0[rows, np.arange(len(rows))] = 1.0
    assert rel_err(got, orc.cheb_moments(H, x0, 64, scale)) <= TOL
    E = np.linspace(-0.3, 0.3, 9)
    sites = [(14, 29, 0), (0, 39, 0)]
    assert rel_err(system.ldos_map(sites, E), system.ldos_map(sites, E, kernel="dict_diag")) <= 1e-10
    assert system._sys.cheb_format()["kernel"] == "dict_diag"
    F = system.free_energy(0.1, cuda=True, vectors=16, moments=512)
    assert system._sys.cheb_format()["kernel"] == "t2"
    assert abs(F - system.free_energy(0.1, cuda=True, vectors=16, moments=512, kernel="dict_diag")) <= 1e-10 * abs(F)
    # where no two-applications-per-pass kernel applies or pays, auto_moments is plain auto (no dictionary / no such lattice; small
    # three-dimensional lattices -- large ones have their own even-vector kernel: tests/test_gpu_cube.py)
    for other, want in ((_periodic(gpu_api, (9, 8, 1), x=False, y=False, random_hop=True), "t2"), (cases.swave_3d(gpu_api, (6, 5, 4)), "dict_diag"),
                        (cases.dwave_rashba(gpu_api, (9, 8, 1)), "t2")):
        other.chebyshev_moments(16, vectors=8, seed=1)
        assert other._sys.cheb_format()["kernel"] == want
    system.chebyshev_moments(16, vectors=4, seed=1)
    assert system._sys.cheb_format()["kernel"] == "t2"         # 1200 sites: four columns are padded to a panel


def test_pair_full_size_junction():
    """C5 (10^6 sites, 8 columns): vectors after 2 x 3 + 1 steps bit-identical to the single-step kernel,
    moments to rounding, mu_0 = 4N exactly, bit-reproducible."""
    import bodge_b200 as b
    from bodge_b200 import workloads

    c = workloads.CONFIGS["C5"]
    system = b.Hamiltonian(b.CubicLattice(c["shape"]))
    assert system.fill(*c["build"](c["shape"])) == 0.0
    scale = system.spectral_bound()
    (cur, prev), fmt = _vectors(system._sys, "pair", 8, 7, scale)
    assert fmt == "pair"
    (want_cur, want_prev), _ = _vectors(system._sys, "dict_diag", 8, 7, scale)
    assert np.array_equal(cur, want_cur) and np.array_equal(prev, want_prev)
    del cur, prev, want_cur, want_prev
    pair = system.chebyshev_moments(40, vectors=8, seed=1234, scale=scale, kernel="pair")
    single = system.chebyshev_moments(40, vectors=8, seed=1234, scale=scale, kernel="dict_diag")
    assert rel_err(pair, single) <= 1e-13
    assert np.array_equal(pair[0], np.full(8, float(system.shape[0])))
    assert np.array_equal(pair, system.chebyshev_moments(40, vectors=8, seed=1234, scale=scale, kernel="pair"))
    t2 = system.chebyshev_moments(40, vectors=8, seed=1234, scale=scale, kernel="t2")
    assert rel_err(t2, single) <= 1e-12
    assert np.array_equal(t2[0], np.full(8, float(system.shape[0])))
    assert np.array_equal(t2, system.chebyshev_moments(40, vectors=8, seed=1234, scale=scale))   # the observables' default
    assert system._sys.cheb_format()["kernel"] == "t2"
