"""The step kernels at full and past-32-bit lattice sizes, site by site, against the extended-precision light-cone
reference of ``lightcone.py`` (CPU twin: ``test_lightcone.py``).

The window blocks are read from the matrix the device holds; the window recursions run over the host cores.  Bounds
are the suite's rounding bounds: ``vc.rounding_ratio <= vc.K_ROUNDING`` for vectors and reads, ``|mu_m - ref_m| <=
64 (m + 1) eps mu_0`` for moments.  No planner switch is set: every plan is the one the planner picks at that size.

* Full-size configurations, 41 probe columns (six panels of eight, the last ragged; eleven of four on the cube kernel):
  every moment ``mu_0 .. mu_{2n-1}`` and ``T_n``, ``T_{n-1}`` in full (``T_n = E_{n/2}`` on the even-vector kernels),
  which must also be exactly zero outside each column's light cone.  Probes sit at the corners, edge midpoints, both
  sides of every seam, the junction's interfaces, flat indices 0, N/2 and N - 1, and on either side of the two-step
  kernels' patch boundaries and of the even segment cuts of x.
* Rademacher columns (pair and single-step kernels) and class columns across a wrap seam, read at single sites through
  the local accumulator with one-hot series.
* Lattices whose element offsets pass 2^31: the vectors of a 3400 x 3400 plane (in double2), the fixed-width matrix copy
  of a 216^3 cube (in doubles).  Skipped, with the numbers, when the device lacks the memory.
* A single rewritten block at a far corner of a 10^6-site matrix must be seen.

Each comparison prints one ``lightcone:`` line with its worst ratios (``pytest -s`` shows them).
"""

import numpy as np
import pytest

import lightcone as lc
import readout_cases as rc
import variant_cases as vc
from bodge_b200 import _native, workloads

pytestmark = pytest.mark.gpu
K = vc.K_ROUNDING
N_COLS = 41
STEPS_2D = 128    # T_n of the probe columns on the 10^6-site planes ...
STEPS_3D = 32     # ... and on the 64^3 cube
STEPS_BIG = 16    # past 32-bit offsets

# config -> kernels asked for (auto_moments = the even-vector kernel where the two-step kernel applies, auto = pair)
FULL = [
    ("C5", ["auto_moments", "auto", "dict_diag", "dict", "ell", "dmma"]),
    ("C5_periodic", ["auto_moments", "auto", "dict_diag", "ell"]),
    ("C5_disordered", ["auto_moments", "auto", "dict_diag", "ell"]),
    ("C5_random", ["auto", "dmma"]),
    ("C5_bilayer", ["auto_moments", "auto", "ell"]),
    ("C4", ["auto_moments", "dict_diag", "dict", "ell", "dmma"]),
]


def report(**fields):
    print("lightcone: " + " ".join(f"{k}={v:.3g}" if isinstance(v, float) else f"{k}={v}" for k, v in fields.items()))


def flat(shape, x, y, z=0):
    return int(z + shape[2] * (y + shape[1] * x))


def pair_patch_starts(M, open_):
    """First owned row of every patch of the two-step kernels on a plane of M rows (``pair_configure``, cheb_pair.cu:
    patches of at most 8 warps x 2 sites - 2 rows, balanced; an open plane's first patch also owns row 0)."""
    p_max = 14
    cover = max(1, M - 2 * open_)
    n_min = -(-cover // p_max)
    P = -(-cover // n_min)
    return [k * P + open_ for k in range(-(-cover // P))]


def probe_sites_2d(shape):
    Lx, Ly, _ = shape
    pts = {(0, 0), (0, Ly - 1), (Lx - 1, 0), (Lx - 1, Ly - 1),                  # corners (flat 0 and N - 1)
           (Lx // 2, 0), (Lx // 2, Ly - 1), (0, Ly // 2), (Lx - 1, Ly // 2),   # edge midpoints = either side of a seam
           (0, Ly // 3), (Lx - 1, Ly // 3), (Lx // 3 + 7, 0), (Lx // 3 + 7, Ly - 1)}
    x1, x2 = Lx // 3, Lx - Lx // 3                                              # junction interfaces (workloads.junction)
    pts |= {(x1 - 1, 2 * Ly // 3), (x1, 2 * Ly // 3), (x2 - 1, Ly // 5), (x2, Ly // 5)}
    starts = pair_patch_starts(Ly, 1)
    for s in (starts[1], starts[len(starts) // 2], starts[-1]):                 # patch boundaries, the last (ragged) one
        pts |= {(Lx // 4 - 1, s - 1), (Lx // 4, s)}
    pts |= {(Lx // 2 - 1, starts[-1] - 1), (3 * Lx // 4, 5)}                   # cuts of 2 and 4 segments of x
    sites = sorted({flat(shape, x, y) for x, y in pts} | {(Lx * Ly) // 2})
    return sites


def probe_sites_3d(shape):
    Lx, Ly, Lz = shape
    e = (0, Lx - 1)
    pts = {(x, y, z) for x in e for y in (0, Ly - 1) for z in (0, Lz - 1)}      # corners
    pts |= {(Lx // 2, Ly // 2, 0), (Lx // 2, 0, Lz // 2), (0, Ly // 2, Lz // 2), (Lx - 1, Ly // 2, Lz - 1)}
    pts |= {(Lx // 3, 7, 8), (Lx // 3, 8, 7), (Lx // 2, 15, 16), (Lx // 2, 31, 32), (2 * Lx // 3, 39, 40)}  # 8x8 patch rims
    return sorted({flat(shape, *p) for p in pts} | {(Lx * Ly * Lz) // 2})


def probe_rows(sites, n_cols=N_COLS):
    """``n_cols`` probe rows cycling over ``sites``, the component advancing every lap and from site to site."""
    S = len(sites)
    rows = [4 * sites[c % S] + (c // S + c % S) % 4 for c in range(n_cols)]
    assert len(set(rows)) == n_cols
    return np.array(rows, dtype=np.int64)


@pytest.fixture(scope="module")
def full():
    """(system, scale, light cone) of one configuration; one large system alive at a time."""
    cache = {}

    def get(key):
        if key not in cache:
            import bodge_b200 as b

            cache.clear()
            _native.release_cached()
            if key is None:
                return None
            c = workloads.CONFIGS[key]
            system = b.Hamiltonian(b.CubicLattice(c["shape"]))
            assert system.fill(*c["build"](c["shape"])) <= 1e-12
            scale = system.spectral_bound()
            cache[key] = (system, scale, lc.Lightcone(c["shape"], system._sys, scale))
        return cache[key]

    yield get
    cache.clear()


def advance_to(sysn, n):
    """Step the recursion to T_n (the even-vector kernels step in twos)."""
    sysn.cheb_steps(n - sysn.cheb_available() // 2)
    assert sysn.cheb_available() // 2 == n


def vector_ratio(got, vectors, which, k):
    """Worst rounding ratio of ``got [4N, C]`` against the window values ``vectors[c][which]``; inf if a column has a
    non-zero outside its light cone."""
    worst = 0.0
    for c, v in enumerate(vectors):
        rows, want = v[0], v[which]
        col = np.ascontiguousarray(got[:, c])
        inside = col[rows]
        if np.count_nonzero(col) != np.count_nonzero(inside):
            return float("inf")
        worst = max(worst, vc.rounding_ratio(inside, want, k))
    return worst


def run_probes(sysn, rows, n, kernel, scale):
    """(format, info, moments, T_n, T_{n-1} or None) of one recursion on probe columns."""
    sysn.cheb_begin(probe_rows=rows, scale=scale, kernel=kernel)
    fmt, info = sysn.cheb_format()["kernel"], sysn.cheb_info()
    advance_to(sysn, n)
    mu = sysn.cheb_read(2 * n, len(rows))
    cur = sysn.cheb_vectors(len(rows), 0)
    prev = None if fmt == "t2" else sysn.cheb_vectors(len(rows), 1)
    sysn.cheb_end()
    return fmt, info, mu, cur, prev


@pytest.mark.parametrize("key,kernels", FULL)
def test_probe_columns_at_full_size(full, monkeypatch, key, kernels):
    vc.set_env(monkeypatch, ())
    system, scale, cone = full(key)
    shape = system.lattice.shape
    n = STEPS_3D if shape[2] > 1 else STEPS_2D
    sites = probe_sites_3d(shape) if shape[2] > 1 else probe_sites_2d(shape)
    rows = probe_rows(sites)
    mu_ref, vectors = cone.run_probes(rows, n)
    seen = set()
    for kernel in kernels:
        fmt, info, mu, cur, prev = run_probes(system._sys, rows, n, kernel, scale)
        seen.add(fmt)
        assert info["n_panels"] == -(-N_COLS // info["panel_width"]) and info["n_panels"] >= 6
        r_mu = rc.worst(rc.moment_ratios(mu, mu_ref))
        r_cur = vector_ratio(cur, vectors, 2, n)
        r_prev = vector_ratio(prev, vectors, 1, n - 1) if prev is not None else 0.0
        del cur, prev
        report(config=key, kernel=kernel, format=fmt, panels=info["n_panels"], n=n, moments=r_mu, T_n=r_cur, T_n1=r_prev)
        assert r_mu <= K, f"{key} {kernel} ({fmt}): moment error {r_mu:.1f} x (m+1) eps mu_0"
        assert r_cur <= K, f"{key} {kernel} ({fmt}): T_{n} error {r_cur:.1f} x (n+1) eps max|T| (inf: non-zero outside the cone)"
        assert r_prev <= K, f"{key} {kernel} ({fmt}): T_{n - 1} error {r_prev:.1f} x n eps max|T|"
    if key in ("C5", "C5_periodic", "C5_disordered"):
        assert {"t2", "pair"} <= seen
    if key == "C4":
        assert "t2" in seen


def local_reads(sysn, begin, coef_len, k, cols, sites):
    """``T_k`` at ``(cols[r], sites[r])`` through the local accumulator with the one-hot series ``e_k``."""
    begin()
    coef = np.zeros(coef_len)
    coef[k] = 1.0
    sysn.cheb_local_begin(coef, cols, sites)
    if k >= 2:
        advance_to(sysn, k)
    fmt = sysn.cheb_format()["kernel"]
    got = sysn.cheb_local_read(len(sites))
    sysn.cheb_end()
    return fmt, got


@pytest.mark.parametrize("kernel", ["auto", "dict_diag", "ell"])
def test_rademacher_reads_at_full_size(full, monkeypatch, kernel):
    vc.set_env(monkeypatch, ())
    system, scale, cone = full("C5")
    shape, sysn = system.lattice.shape, system._sys
    seed, n_cols = 4321, 8
    sites = np.array((probe_sites_2d(shape) * 4)[:64], dtype=np.int64)
    rng = np.random.default_rng(1)
    sites[-16:] = rng.integers(0, system.lattice.size, 16)
    cols = np.arange(len(sites)) % n_cols
    ks = (1, 2, 31, 64)
    want = cone.run_reads(lambda rows, c: lc.rademacher_rows(seed, rows, c), cols, sites, ks)
    for k in ks:
        fmt, got = local_reads(sysn, lambda: sysn.cheb_begin(n_random=n_cols, seed=seed, scale=scale, kernel=kernel),
                               k + 1, k, cols, sites)
        ratio = vc.rounding_ratio(got, want[k], k)
        report(config="C5", start="rademacher", kernel=kernel, format=fmt, k=k, reads=ratio)
        assert ratio <= K, f"{kernel} ({fmt}): T_{k} reads, error {ratio:.1f} x (k+1) eps max|T|"


def test_class_reads_across_the_wrap_seam(full, monkeypatch):
    vc.set_env(monkeypatch, ())
    system, scale, cone = full("C5_periodic")
    shape, sysn = system.lattice.shape, system._sys
    Lx, Ly, _ = shape
    spacing = 7                       # does not divide 1000: the last run of each axis is longer
    assert Lx % spacing and system._wrapping_axes() == (True, True, False)
    site_class = system._classes(spacing)
    pts = [(0, 0), (Lx - 1, 0), (0, Ly - 1), (Lx - 1, Ly - 1), (1, 400), (Lx - 2, 400), (0, 401), (Lx - 1, 401),
           (500, 0), (500, Ly - 1), (501, 1), (501, Ly - 2), (Lx - 1, 997), (0, 3), (333, 333), (Lx // 3, 2)]
    sites = np.array([flat(shape, x, y) for x, y in pts], dtype=np.int64)
    class_rows = 4 * site_class[sites].astype(np.int64) + np.arange(len(sites)) % 4
    cols = np.arange(len(sites))
    ks = (2, 9, 32)
    want = cone.run_reads(lambda rows, c: lc.class_start(site_class, rows, class_rows[np.asarray(c)]), cols, sites, ks)
    for k in ks:
        fmt, got = local_reads(sysn, lambda: sysn.cheb_begin(class_rows=class_rows, scale=scale, kernel="auto"),
                               k + 1, k, cols, sites)
        ratio = vc.rounding_ratio(got, want[k], k)
        report(config="C5_periodic", start="class", spacing=spacing, format=fmt, k=k, reads=ratio)
        assert ratio <= K, f"class columns ({fmt}): T_{k} reads, error {ratio:.1f} x (k+1) eps max|T|"


def test_a_rewritten_corner_block_is_seen(full, monkeypatch):
    """Negative control: one on-site block at the far corner of C5 is changed by 1e-9 after the reference has gathered
    its window.  The comparison must fail; with the block restored it passes again."""
    vc.set_env(monkeypatch, ())
    system, scale, cone = full("C5")
    sysn = system._sys
    N = system.lattice.size
    s, n = N - 1, 16
    rows = np.array([4 * s + b for b in range(4)] + [4 * (s - 1) + b for b in range(4)], dtype=np.int64)
    mu_ref, vectors = cone.run_probes(rows, n)
    h = sysn.gather_blocks(sysn.lookup([s], [s]))[0][:2, :2].copy()
    none = np.empty((0, 2, 2), dtype=np.complex128)
    sysn.scatter([s], [s], [h + 1e-9 * np.diag([1.0, -1.0])], [], [], none)
    try:
        _, _, mu, cur, _ = run_probes(sysn, rows, n, "auto", scale)
    finally:
        sysn.scatter([s], [s], [h], [], [], none)
    r_bad = max(vector_ratio(cur, vectors, 2, n), rc.worst(rc.moment_ratios(mu, mu_ref)))
    _, _, mu, cur, _ = run_probes(sysn, rows, n, "auto", scale)
    r_good = max(vector_ratio(cur, vectors, 2, n), rc.worst(rc.moment_ratios(mu, mu_ref)))
    report(config="C5", control="corner block +1e-9", changed=r_bad, restored=r_good)
    assert r_bad > K, f"a changed block went unseen (ratio {r_bad:.1f})"
    assert r_good <= K


# name -> (shape, builder, kernels)
BIG = {
    "plane_3400": ((3400, 3400, 1), workloads.readme_swave, ["dict_diag", "t2"]),
    "cube_216": ((216, 216, 216), workloads.swave_3d, ["ell", "dmma"]),
}


@pytest.mark.parametrize("name", list(BIG))
def test_past_32_bit_offsets(full, monkeypatch, name):
    import torch

    import bodge_b200 as b

    vc.set_env(monkeypatch, ())
    full(None)  # no other system alive
    shape, build, kernels = BIG[name]
    N = int(np.prod(shape))
    dims = sum(1 for L in shape if L > 1)
    n_blocks = (1 + 2 * dims) * N
    vec_bytes = 4 * N * 48 * 16                   # 41 columns in six 8-column panels, double2
    # offsets past 2^31: the plane's vectors in double2 elements, the cube's fixed-width copy in doubles
    assert max(vec_bytes // 16, n_blocks * 32) >= 2**31
    need = 2 * vec_bytes + 4 * n_blocks * 256      # two vectors; skeleton, compacted and kernel-native copies of the blocks
    free, total = torch.cuda.mem_get_info()
    report(lattice=name, sites=N, free_GB=free / 1e9, total_GB=total / 1e9, estimate_GB=need / 1e9)
    if free < need:
        pytest.skip(f"{name}: needs about {need / 1e9:.0f} GB (vectors {2 * vec_bytes / 1e9:.0f} GB, blocks "
                    f"{4 * n_blocks * 256 / 1e9:.0f} GB), {free / 1e9:.0f} GB of {total / 1e9:.0f} GB free")
    system = b.Hamiltonian(b.CubicLattice(shape))
    try:
        assert system.fill(*build(shape)) <= 1e-12
        sysn, scale = system._sys, system.spectral_bound()
        cone = lc.Lightcone(shape, sysn, scale)
        Lx, Ly, Lz = shape
        far = {N - 1 - d for d in range(0, 9 * Lz * Ly, Ly * Lz + Lz + 1)} | {N - 1 - d for d in range(6)}
        far |= {flat(shape, Lx - 1, 0, Lz - 1), flat(shape, Lx - 1, Ly - 1, 0), flat(shape, Lx - 2, Ly - 1, Lz - 1)}
        sites = sorted(far)
        rows = probe_rows(sites)
        n = STEPS_BIG
        mu_ref, vectors = cone.run_probes(rows, n)
        # reads of T_n at each column's own site and one hop lower in x
        cols = np.concatenate([np.arange(N_COLS)] * 2)
        read_sites = np.concatenate([rows // 4, rows // 4 - Ly * Lz])
        want = np.stack([vectors[c][2].reshape(-1, 4)[lc.local_index(vectors[c][0][::4] // 4, s)] for c, s in
                         zip(cols, read_sites)])
        for kernel in kernels:
            sysn.cheb_begin(probe_rows=rows, scale=scale, kernel=kernel)
            fmt = sysn.cheb_format()["kernel"]
            local = fmt != "t2"
            if local:
                coef = np.zeros(n + 1)
                coef[n] = 1.0
                sysn.cheb_local_begin(coef, cols, read_sites)
            advance_to(sysn, n)
            mu = sysn.cheb_read(2 * n, N_COLS)
            got = sysn.cheb_local_read(len(cols)) if local else None
            used = sysn.device_bytes()
            sysn.cheb_end()
            r_mu = rc.worst(rc.moment_ratios(mu, mu_ref))
            r_reads = vc.rounding_ratio(got, want, n) if local else 0.0
            report(lattice=name, kernel=kernel, format=fmt, n=n, moments=r_mu, reads=r_reads, device_GB=used / 1e9)
            assert r_mu <= K, f"{name} {kernel}: moment error {r_mu:.1f} x (m+1) eps mu_0"
            assert r_reads <= K, f"{name} {kernel}: T_{n} reads, error {r_reads:.1f} x (n+1) eps max|T|"
    finally:
        system._sys.close()
        del system
        _native.release_cached()
