"""The Chebyshev read-outs against an extended-precision reference (``readout_cases``), at the recursion lengths the
observables run.

* Moments of every stepping (single-step kernels, pair, even-vector on an open and a periodic plane and on a cube), for
  1, 3, 13 and 41 columns, each moment on its own: ``|mu_n - ref_n| <= K (n + 1) eps mu_0``.  The reads run across the
  growths of the dot rows (every read is the bitwise prefix of the last).
* ``kpm_resolvent`` at |w| -> 1, ``kpm_contract`` / ``sum_columns`` past one warp, the local accumulator over series of
  4096 terms.
* Device-pointer outputs and a borrowed stream give the bits of the host outputs.
* Per-column moments with ``n_moments * n_cols >= 2^31`` (64-bit index of ``moments_from_dots``).
"""

import ctypes as C

import numpy as np
import pytest

import readout_cases as rc
import variant_cases as vc
from bodge_b200 import _native
from bodge_b200.kpm import resolvent_weights
from oracle import bdg_oracle as orc

pytestmark = pytest.mark.gpu
SEED = 5
K = vc.K_ROUNDING
LONG_COLS = [0, 1, 2, 12, 40]   # columns the 32768-moment reference carries: the last of 1, 3, 13 and 41 columns, and one more

# geometry -> (lattice shape, periodic in-plane, model)
GEOMETRIES = {
    "plane": ((6, 5, 1), False, "diag"),
    "plane_gen": ((6, 5, 1), False, "gen"),
    "torus": ((6, 5, 1), True, "diag"),
    "cube": ((3, 4, 5), False, "diag"),
}
# stepping -> (geometry, kernel, environment, kernel cheb_format must report)
STEPPINGS = {
    "dict_diag": ("plane", "dict_diag", (), "dict_diag"),
    "dict": ("plane_gen", "dict", (), "dict"),
    "ell": ("plane_gen", "ell", (), "ell"),
    "dmma": ("plane_gen", "dmma", (), "dmma"),
    "fma": ("plane_gen", "fma", (), "fma"),
    "pair": ("plane", "pair", (), "pair"),
    "t2_open": ("plane", "t2", (), "t2"),
    "t2_torus": ("torus", "t2", (), "t2"),
    "t2_cube": ("cube", "t2", (("BDG_CUBE_SHAPE", 1),), "t2"),
}
LENGTHS = list(range(1, 9)) + [2000] + list(range(2046, 2053)) + [4100, 32768]
SHORT = 4100   # moments of the all-column reference


@pytest.fixture(scope="module")
def world(gpu_api):
    """Per geometry: the system, its scale and the references, computed once per module on demand."""
    systems, refs = {}, {}

    def system(geometry):
        if geometry not in systems:
            shape, torus, model = GEOMETRIES[geometry]
            lattice = gpu_api.CubicLattice(shape)
            pairs = vc.periodic_pairs(lattice) if torus else list(lattice.bonds())
            h = vc.fill(gpu_api, gpu_api.Hamiltonian(lattice), pairs, model)
            scale = h.spectral_bound()
            systems[geometry] = (h, scale, rc.ScalarReference(*h._sys.export_bsr(True), scale))
        return systems[geometry]

    def moments(geometry, cols, n_moments):
        """Reference moments ``[n_moments, len(cols)]`` of the Rademacher columns ``cols``."""
        key = (geometry, tuple(cols), n_moments)
        if key not in refs:
            h, _, ref = system(geometry)
            x0 = orc.rademacher(SEED, 4 * h._sys.n_sites, np.asarray(cols))
            refs[key] = rc.reference_readouts(ref, x0, n_moments)[0]
        return refs[key]

    yield system, moments
    for h, _, _ in systems.values():
        h._sys.cheb_end()
    _native.release_cached(0)


def begin(world, monkeypatch, stepping, n_cols, **kw):
    system, _ = world
    geometry, kernel, env, expect = STEPPINGS[stepping]
    h, scale, _ = system(geometry)
    vc.set_env(monkeypatch, env)
    h._sys.cheb_begin(n_random=n_cols, seed=SEED, scale=scale, kernel=kernel, **kw)
    assert h._sys.cheb_format()["kernel"] == expect
    return h._sys


def step_to(sysn, n_moments):
    """Step until ``n_moments`` moments are available."""
    need = (n_moments + 1) // 2 - 1 - (sysn.cheb_available() // 2 - 1)
    if need > 0:
        sysn.cheb_steps(need)


def check_moments(got, want, label, even_vectors):
    ratios = rc.moment_ratios(got, want)
    if even_vectors:
        msg = f"{label}: worst even {rc.worst(ratios, 0):.2f}, odd {rc.worst(ratios, 1):.2f} x (n+1) eps mu_0 (bound {K})"
    else:
        msg = f"{label}: worst {rc.worst(ratios):.2f} x (n+1) eps mu_0 (bound {K})"
    assert rc.worst(ratios) <= K, msg
    return ratios


# ---- moments per stepping ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_cols", [1, 3, 13, 41])
@pytest.mark.parametrize("stepping", sorted(STEPPINGS))
def test_moments_per_stepping_and_length(world, monkeypatch, stepping, n_cols):
    system, moments = world
    geometry = STEPPINGS[stepping][0]
    sysn = begin(world, monkeypatch, stepping, n_cols)
    even = stepping.startswith("t2")
    reads = []
    for m in LENGTHS:
        step_to(sysn, m)
        reads.append(sysn.cheb_read(m, n_cols))
    summed = sysn.cheb_read(LENGTHS[-1], n_cols, summed=True)
    sysn.cheb_end()
    last = reads[-1]
    for m, got in zip(LENGTHS, reads):   # reads across the growths of the dot rows: earlier reads are prefixes
        assert np.array_equal(got, last[:m]), f"the read of {m} moments is not the prefix of the last read"
    short = moments(geometry, tuple(range(41)), SHORT)[:, :n_cols]
    for m, got in zip(LENGTHS[:-1], reads[:-1]):
        check_moments(got, short[:m], f"{stepping}, {n_cols} columns, {m} moments", even)
    cols = [c for c in LONG_COLS if c < n_cols]
    want = moments(geometry, tuple(LONG_COLS), LENGTHS[-1])[:, : len(cols)]
    check_moments(last[:, cols], want, f"{stepping}, {n_cols} columns, {LENGTHS[-1]} moments", even)
    assert np.max(np.abs(summed - last.sum(axis=1))) <= 1e-13 * n_cols * np.max(np.abs(last[0]))


T2_LONG = 131072


@pytest.mark.parametrize("stepping", ["t2_open", "t2_torus", "t2_cube"])
def test_t2_odd_moments_over_a_long_recursion(world, monkeypatch, stepping):
    """The even-vector recursion's odd moments come from a two-term recurrence along the launches (t2_normalize); its
    error, per moment against the extended-precision recursion, stays within the bound of the single-step kernels."""
    _, moments = world
    sysn = begin(world, monkeypatch, stepping, 2)
    marks = (2048, 32768, T2_LONG)
    reads = {}
    for m in marks:
        step_to(sysn, m)
        reads[m] = sysn.cheb_read(m, 2)
    sysn.cheb_end()
    want = moments(STEPPINGS[stepping][0], (0, 1), T2_LONG)
    report = []
    for m in marks:
        assert np.array_equal(reads[m], reads[T2_LONG][:m])
        r = rc.moment_ratios(reads[m], want[:m])
        report.append(f"{m}: even {rc.worst(r, 0):.2f} odd {rc.worst(r, 1):.2f}")
    print(f"\n{stepping} worst ratio to (n+1) eps mu_0 at " + ", ".join(report))
    r = rc.moment_ratios(reads[T2_LONG], want)
    assert rc.worst(r) <= K, f"{stepping}: " + ", ".join(report)


# ---- kpm_resolvent --------------------------------------------------------------------------------------------------------
def _edge_energies():
    out = []
    for re in (0.0, 0.999, -0.999):
        for im in (0.1, 1e-2, 1e-3, 1e-4):
            out += [complex(re, im), complex(re, -im)]
    return np.array(out)


def _moments_for(w, tol=1e-13):
    return int(np.ceil(np.log(tol) / np.log(np.max(np.abs(w)))))


def check_resolvent(sysn, n_moments, n_cols, z, cols):
    w, pref = resolvent_weights(z)
    got = sysn.kpm_resolvent(n_moments, n_cols, w, pref)
    mu = sysn.cheb_read(n_moments, n_cols)          # the moments the kernel sums, bit for bit
    want, size = rc.resolvent(mu[:, cols], w, pref)
    ratio = float(np.max(np.abs(got[cols].astype(np.clongdouble) - want) / ((n_moments + 1) * rc.EPS * size)))
    assert ratio <= K, f"{n_moments} moments, {len(z)} energies: error {ratio:.2f} x (N+1) eps sum|terms|"
    again = sysn.kpm_resolvent(n_moments, n_cols, w, pref)
    assert np.array_equal(again, got)
    return got


def test_resolvent_as_w_approaches_the_unit_circle(world, monkeypatch):
    z = _edge_energies()
    w, _ = resolvent_weights(z)
    n_moments = _moments_for(w) | 1
    assert np.max(np.abs(w)) ** n_moments < 1e-13 and n_moments <= 1 << 20
    sysn = begin(world, monkeypatch, "t2_open", 41)
    step_to(sysn, n_moments)
    check_resolvent(sysn, n_moments, 41, z, [0, 12, 40])
    sysn.cheb_end()


@pytest.mark.parametrize("n_cols", [1, 13, 41])
def test_resolvent_counts(world, monkeypatch, n_cols):
    rng = np.random.default_rng(n_cols)
    z7 = rng.uniform(-0.999, 0.999, 7) + 1j * rng.choice([-1, 1], 7) * rng.uniform(1e-3, 0.1, 7)
    z1000 = np.linspace(-0.999, 0.999, 1000) + 1j * np.where(np.arange(1000) % 2, 0.01, -0.01)
    n_long = _moments_for(resolvent_weights(z1000)[0]) | 1
    sysn = begin(world, monkeypatch, "dict_diag", n_cols)
    step_to(sysn, max(n_long, 2047))
    cols = sorted({0, n_cols // 2, n_cols - 1})
    for n_moments in (1, 2, 2047):
        for z in (z7[:1], z7):
            check_resolvent(sysn, n_moments, n_cols, z, list(range(n_cols)))
    check_resolvent(sysn, n_long, n_cols, z1000, cols)
    sysn.cheb_end()


# ---- kpm_contract, sum_columns -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_cols", [1, 31, 32, 33, 41, 100])
def test_contraction_and_column_sum(world, monkeypatch, n_cols):
    sysn = begin(world, monkeypatch, "dict_diag", n_cols)
    step_to(sysn, 32768)
    rng = np.random.default_rng(n_cols)
    mu = sysn.cheb_read(32768, n_cols)
    for n_moments in (1, 2, 31, 32, 33, 32768):
        coef = rng.uniform(-1.0, 1.0, n_moments) / np.arange(1, n_moments + 1)
        got = sysn.kpm_contract(coef, n_cols)
        want, size = rc.contract(mu[:n_moments], coef)
        ratio = float(np.max(np.abs(got.astype(np.longdouble) - want) / ((n_moments + 1) * rc.EPS * size)))
        assert ratio <= K, f"{n_moments} moments: error {ratio:.2f} x (N+1) eps sum|c mu|"
        total = sysn.kpm_contract(coef, n_cols, summed=True)
        assert total == rc.warp_sum(got), f"{n_moments} moments: the summed contraction is not the sum of the columns"
        assert np.array_equal(sysn.kpm_contract(coef, n_cols), got) and sysn.kpm_contract(coef, n_cols, summed=True) == total
    sysn.cheb_end()


# ---- local accumulator, long series --------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_coef", [4095, 4096])
@pytest.mark.parametrize("stepping", ["pair", "dict_diag"])
def test_local_accumulator_over_a_long_series(world, monkeypatch, stepping, n_coef):
    system, _ = world
    h, scale, ref = system("plane")
    n_cols, n_sites = 41, h._sys.n_sites
    rng = np.random.default_rng(n_coef)
    coef = rng.uniform(-1.0, 1.0, n_coef)
    cols = np.concatenate([rng.integers(0, n_cols, 40), [n_cols - 1, n_cols - 1, 40, 33]])
    sites = np.concatenate([rng.integers(0, n_sites, 40), [n_sites - 1, n_sites - 1, 0, 7]])
    cols, sites = np.append(cols, cols[0]), np.append(sites, sites[0])   # duplicate reads
    sysn = begin(world, monkeypatch, stepping, n_cols)
    sysn.cheb_local_begin(coef, cols, sites)
    sysn.cheb_steps(n_coef)   # past the end of the series
    got = sysn.cheb_local_read(len(cols))
    sysn.cheb_end()
    rows = (4 * sites[:, None] + np.arange(4)).ravel()
    x0 = orc.rademacher(SEED, 4 * n_sites, np.arange(n_cols))
    _, terms, t_max = rc.reference_readouts(ref, x0, 1, local=(rows, np.repeat(cols, 4), n_coef))
    want = rc.local_sums(terms, coef)[0].reshape(-1, 4)
    bound = n_coef * rc.EPS * max(1.0, t_max) * np.sum(np.abs(coef))
    ratio = float(np.max(np.abs(got.astype(np.clongdouble) - want))) / bound
    assert ratio <= K, f"{stepping}, {n_coef} terms: error {ratio:.2f} x the rounding bound"
    assert np.array_equal(got[-1], got[0]) and np.array_equal(got[40], got[41])


# ---- device outputs, borrowed stream -------------------------------------------------------------------------------------
def _device_reads(torch, sysn, dev, n_cols, n_moments, coef, w, pref, n_reads):
    """Every read-out once with a device pointer: per-column and summed moments, resolvent, per-column and summed
    contraction, local sums."""
    lib = _native.load()
    out = {
        "mu": torch.empty((n_moments, n_cols), dtype=torch.float64, device=dev),
        "mu_sum": torch.empty(n_moments, dtype=torch.float64, device=dev),
        "g": torch.empty((n_cols, len(w)), dtype=torch.complex128, device=dev),
        "f": torch.empty(n_cols, dtype=torch.float64, device=dev),
        "f_sum": torch.empty(1, dtype=torch.float64, device=dev),
        "local": torch.empty((n_reads, 4), dtype=torch.complex128, device=dev),
    }
    sysn.cheb_read(n_moments, n_cols, device_ptr=out["mu"].data_ptr())
    sysn.cheb_read(n_moments, n_cols, summed=True, device_ptr=out["mu_sum"].data_ptr())
    wp, pp = np.ascontiguousarray(w), np.ascontiguousarray(pref)
    _native.check(lib.bdg_kpm_resolvent(sysn._h, n_moments, len(w), wp.ctypes.data_as(C.c_void_p),
                                        pp.ctypes.data_as(C.c_void_p), C.c_void_p(out["g"].data_ptr()), 1))
    cp = np.ascontiguousarray(coef)
    for key, reduce in (("f", 0), ("f_sum", 1)):
        _native.check(lib.bdg_kpm_contract(sysn._h, len(coef), cp.ctypes.data_as(C.c_void_p), reduce,
                                           C.c_void_p(out[key].data_ptr()), 1))
    sysn.cheb_local_read(n_reads, device_ptr=out["local"].data_ptr())
    return out


def _host_reads(sysn, n_cols, n_moments, coef, w, pref, n_reads):
    return {"mu": sysn.cheb_read(n_moments, n_cols), "mu_sum": sysn.cheb_read(n_moments, n_cols, summed=True),
            "g": sysn.kpm_resolvent(n_moments, n_cols, w, pref), "f": sysn.kpm_contract(coef, n_cols),
            "f_sum": np.array([sysn.kpm_contract(coef, n_cols, summed=True)]), "local": sysn.cheb_local_read(n_reads)}


def test_device_outputs_and_a_borrowed_stream(world, monkeypatch):
    import torch

    system, _ = world
    h, _, _ = system("plane")
    dev = f"cuda:{h.device}"
    n_cols, n_moments = 13, 301
    rng = np.random.default_rng(3)
    coef = rng.uniform(-1.0, 1.0, n_moments)
    w, pref = resolvent_weights(np.array([0.3 + 0.05j, -0.7 - 0.01j, 0.0 + 0.2j]))
    cols, sites = np.array([0, 12, 12, 5]), np.array([0, 29, 29, 17])
    sysn = begin(world, monkeypatch, "pair", n_cols)
    sysn.cheb_local_begin(coef[:200], cols, sites)
    step_to(sysn, n_moments)
    host = _host_reads(sysn, n_cols, n_moments, coef, w, pref, len(cols))
    got = _device_reads(torch, sysn, dev, n_cols, n_moments, coef, w, pref, len(cols))
    torch.cuda.synchronize(dev)
    for key, value in got.items():
        assert np.array_equal(value.cpu().numpy(), host[key]), key

    stream = torch.cuda.Stream(device=dev)
    sysn.set_stream(stream.cuda_stream)
    try:
        sysn.cheb_steps(100)   # the recursion goes on on the borrowed stream
        n_more = n_moments + 200
        with torch.cuda.stream(stream):
            got = _device_reads(torch, sysn, dev, n_cols, n_more, coef, w, pref, len(cols))
        stream.synchronize()
        host = _host_reads(sysn, n_cols, n_more, coef, w, pref, len(cols))
        for key, value in got.items():
            assert np.array_equal(value.cpu().numpy(), host[key]), f"{key} on the borrowed stream"
    finally:
        sysn.set_stream(None)
    sysn.cheb_steps(1)
    assert np.array_equal(sysn.cheb_read(n_moments, n_cols), host["mu"][:n_moments])
    sysn.cheb_end()


# ---- 64-bit flat index of moments_from_dots ------------------------------------------------------------------------------
def test_per_column_moments_past_two_to_the_31(gpu_api):
    """32768 probe columns x 65536 moments = 2^31 outputs: the per-column read on device output must write every one."""
    import torch

    free, _ = torch.cuda.mem_get_info(0)
    if free < 48e9:
        pytest.skip(f"needs about 48 GB of free device memory, {free / 1e9:.0f} GB free")
    lattice = gpu_api.CubicLattice((8, 1, 1))
    h = vc.fill(gpu_api, gpu_api.Hamiltonian(lattice), list(lattice.bonds()), "diag")
    scale = h.spectral_bound()
    sysn = h._sys
    n_cols, n_moments, rows = 32768, 65536, 32
    assert n_cols * n_moments >= 1 << 31
    sysn.cheb_begin(probe_rows=np.arange(rows), scale=scale, kernel="dict_diag")
    sysn.cheb_steps(n_moments // 2 - 1)
    want = sysn.cheb_read(n_moments, rows)
    sysn.cheb_end()
    out = None
    try:
        sysn.cheb_begin(probe_rows=np.arange(n_cols) % rows, scale=scale, kernel="dict_diag")
        sysn.cheb_steps(n_moments // 2 - 1)
        out = torch.full((n_moments, n_cols), float("nan"), dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize(0)   # the fill runs on torch's stream, the read on the library's
        sysn.cheb_read(n_moments, n_cols, device_ptr=out.data_ptr())
        torch.cuda.synchronize(0)
        for first in (0, n_cols // 2, n_cols - rows):
            got = out[:, first:first + rows].cpu().numpy()
            assert not np.isnan(got).any(), f"columns {first}..{first + rows - 1} were not written"
            assert np.max(np.abs(got - want)) <= 1e-12, f"columns {first}..{first + rows - 1} differ from the 32-column run"
    finally:
        del out
        sysn.cheb_end()
        torch.cuda.empty_cache()
        _native.release_cached(0)
