"""In-place patches of the step kernels' copies (``csrc/formats.cu``: ``ell_patch`` / ``patch_blocks``) against a fresh
build and an extended-precision reference, after every step of the scripted sequences of ``patch_cases``.

After each scatter:

1. **path** -- ``bdg_stats`` moves as the step's label says, read at the first ``cheb_begin`` (where a rebuild runs);
2. **twin** -- a system built fresh from the patched system's skeleton data exports the same BSR and CSR arrays and the
   same norm, bit for bit;
3. **eligibility** -- both accept the same kernel names (the patched dictionary keeps stale entries, so on 3-D lattices it
   may refuse ``t2`` past 64 distinct blocks), and, read off the exported blocks alone: a DIAG instantiation runs only
   when every off-site block is real-diagonal, an SD instantiation only when every on-site block is;
4. **values** -- every accepted kernel's T_n and T_{n-1} after 7 steps on 13 columns are within rounding of the
   ``np.clongdouble`` recursion, its moments equal the oracle's to 1e-10 (Hermitian states: the library doubles the
   moments from T_n, which assumes H = H^†), and where the twin launched the same instantiations all of it is bit for bit
   the twin's.  ``pair`` / ``t2`` run with ``BDG_PAIR_SELF`` 0 and 1, so that stale dictionary entries cannot send the
   two systems to different instantiations.
"""

import numpy as np
import pytest

import patch_cases as pc
import variant_cases as vc
from oracle import bdg_oracle as orc
from util import rel_err, same_bits

pytestmark = pytest.mark.gpu
SEED = 13
N_COLS = 13
STEPS = 7
CUBE_MAX_UNIQUE = 64   # distinct blocks the 3-D even-vector kernel holds (kCubeMaxUnique)


def _kernel_flags(name):
    """(DIAG, SD) of an instantiation: real-diagonal hopping / real-diagonal on-site products."""
    family, args = name.split("<", 1)
    args = [a.strip() for a in args.rstrip(">").split(",")]
    if family == "cheb_step_ell":
        return args[4] == "true", args[5] == "true"
    if family == "cheb_pair_step":
        return args[0] == "true", args[3] == "true"
    return family == "cheb_cube_step", False


def _run(sysn, scale, kernel, n_cols):
    """One forced recursion of STEPS steps, or None when ``cheb_begin`` refuses the kernel."""
    try:
        sysn.cheb_begin(n_random=n_cols, seed=SEED, scale=scale, kernel=kernel)
    except ValueError:
        return None
    fmt = sysn.cheb_format()
    sysn.cheb_steps(STEPS)
    n = sysn.cheb_available() // 2
    out = dict(launched=vc.short_names(sysn.cheb_launched()), n=n, cur=sysn.cheb_vectors(n_cols, 0),
               prev=None if fmt["kernel"] == "t2" else sysn.cheb_vectors(n_cols, 1), mu=sysn.cheb_read(2 * n, n_cols))
    return out   # (no cheb_end: it releases the copies the next scatter is to patch)


def _runs(system, scale, monkeypatch, n_cols):
    """Every kernel name of the library (pair / t2 once per BDG_PAIR_SELF) -> run or None."""
    from bodge_b200 import _native

    out = {}
    for kernel in _native.KERNELS:
        for env in ((("BDG_PAIR_SELF", 0),), (("BDG_PAIR_SELF", 1),)) if kernel in ("pair", "t2") else ((),):
            vc.set_env(monkeypatch, env)
            out[kernel, env] = _run(system._sys, scale, kernel, n_cols)
    vc.set_env(monkeypatch, ())
    return out


class _Reference:
    """T_n of the extended-precision recursion and the oracle's moments over the exported matrix, computed once."""

    def __init__(self, bsr, scale, n_cols):
        self.ref = vc.Reference(*bsr, scale)
        self.H = orc.to_scipy(*bsr)
        self.scale = scale
        self.x0 = orc.rademacher(SEED, self.H.shape[0], np.arange(n_cols))
        self.T, self.mu = [], None

    def vectors(self, n):
        if len(self.T) <= n:
            self.T = self.ref.vectors(self.x0, n)
        return self.T

    def moments(self, m):
        if self.mu is None or len(self.mu) < m:
            self.mu = orc.cheb_moments(self.H, self.x0, m, self.scale)
        return self.mu[:m]


def _check_copies(gpu_api, system, monkeypatch, hermitian, allowed_refusals, n_cols, where):
    """Points 2-4 of the module docstring for the current state of ``system``."""
    sysn = system._sys
    twin = gpu_api.Hamiltonian(system.lattice, device=system.device)
    twin._data = np.asarray(system._data)
    bsr, csr = sysn.export_bsr(True), sysn.export_csr()
    for a, b in zip(bsr, twin._sys.export_bsr(True)):
        assert same_bits(a, b), f"{where}: BSR export differs from a fresh build"
    for a, b in zip(csr, twin._sys.export_csr()):
        assert same_bits(a, b), f"{where}: CSR export differs from a fresh build"
    assert sysn.norm_inf() == twin._sys.norm_inf(), where
    scale = system.spectral_bound()

    indptr, indices, data = bsr
    offsite_diag = pc.offsite_real_diagonal(indptr, indices, data)
    onsite_diag = pc.onsite_real_diagonal(indptr, indices, data)
    ref = _Reference(bsr, scale, n_cols)
    got, want = _runs(system, scale, monkeypatch, n_cols), _runs(twin, scale, monkeypatch, n_cols)
    for key, run in got.items():
        tag = f"{where} {key[0]}{''.join(f' {k}={v}' for k, v in key[1])}"
        if run is None:
            assert want[key] is None or key[0] in allowed_refusals, f"{tag}: refused, a fresh build accepts it"
            continue
        assert want[key] is not None, f"{tag}: accepted, a fresh build refuses it"
        for name in run["launched"]:
            diag, sd = _kernel_flags(name)
            assert offsite_diag or not diag, f"{tag}: {name} runs with off-site blocks that are not real-diagonal"
            assert onsite_diag or not sd, f"{tag}: {name} runs with on-site blocks that are not real-diagonal"
        n = run["n"]
        T = ref.vectors(n)
        ratio = vc.rounding_ratio(run["cur"], T[n], n)
        assert ratio <= vc.K_ROUNDING, f"{tag}: T_{n} off by {ratio:.3g} x the rounding bound"
        if run["prev"] is not None:
            ratio = vc.rounding_ratio(run["prev"], T[n - 1], n - 1)
            assert ratio <= vc.K_ROUNDING, f"{tag}: T_{n - 1} off by {ratio:.3g} x the rounding bound"
        if hermitian:
            assert rel_err(run["mu"], ref.moments(2 * n)) <= 1e-10, f"{tag}: moments differ from the oracle"
        if want[key]["launched"] == run["launched"]:
            assert np.array_equal(run["cur"], want[key]["cur"]), f"{tag}: T_n differs from a fresh build"
            assert (run["prev"] is None) or np.array_equal(run["prev"], want[key]["prev"]), f"{tag}: T_n-1 differs"
            assert np.array_equal(run["mu"], want[key]["mu"]), f"{tag}: moments differ from a fresh build"
    twin._sys.close()
    return got


def _begin_stats(sysn):
    """``bdg_stats`` and the distinct blocks after the first ``cheb_begin`` (which runs a pending rebuild)."""
    sysn.cheb_begin(n_random=N_COLS, seed=SEED, scale=1.0, kernel="auto")
    distinct = sysn.cheb_format()["distinct_blocks"]
    return sysn.stats(), distinct


@pytest.mark.parametrize("geometry,model", pc.SEQUENCES, ids=[f"{g}-{m}" for g, m in pc.SEQUENCES])
def test_patched_copies_after_every_step(gpu_api, monkeypatch, geometry, model):
    seq = pc.sequence(geometry, model)
    system = vc.build(gpu_api, geometry, model)
    sysn = system._sys
    ptr, idx, dat = orc.eliminate_zeros(seq.indptr, seq.indices, seq.initial)
    bsr = sysn.export_bsr(True)
    assert np.array_equal(bsr[0], ptr) and np.array_equal(bsr[1], idx) and same_bits(bsr[2], dat)
    stats, distinct = _begin_stats(sysn)
    verified = True
    three_d = geometry in ("slab", "cube3d")
    for step in seq.steps:
        where = f"{step.name} ({step.path})"
        if step.hermitian:
            system.fill(*step.packed)
        else:  # the listed check raises; the matrix and its copies keep the write, as in the reference
            with pytest.raises(RuntimeError):
                system.fill(*step.packed)
        now, now_distinct = _begin_stats(sysn)
        d = {k: now[k] - stats[k] for k in now}
        if step.path == "patch":
            assert d["patched_scatters"] == 1 and d["patched_blocks"] == step.n_written, f"{where}: {d}"
            assert d["native_builds"] == 0 and d["compactions"] == 0, f"{where}: {d}"
        else:
            assert d["patched_scatters"] == 0 and d["patched_blocks"] == 0, f"{where}: {d}"
            assert d["native_builds"] == 1 and d["compactions"] == 1, f"{where}: {d}"
        assert d["listed_hermitian_checks"] == (1 if verified else 0), f"{where}: {d}"
        if not seq.dictionary:
            assert now_distinct == 0, where
        elif step.new_entries is not None:
            assert now_distinct == distinct + step.new_entries, f"{where}: {distinct} -> {now_distinct} distinct blocks"
        stats, distinct, verified = now, now_distinct, step.hermitian

        ptr, idx, dat = orc.eliminate_zeros(seq.indptr, seq.indices, step.data)
        bsr = sysn.export_bsr(True)
        assert np.array_equal(bsr[0], ptr) and np.array_equal(bsr[1], idx) and same_bits(bsr[2], dat), \
            f"{where}: the exported matrix is not the oracle's"
        allowed = ("t2",) if three_d and distinct > CUBE_MAX_UNIQUE else ()
        _check_copies(gpu_api, system, monkeypatch, step.hermitian, allowed, N_COLS, where)


def test_dictionary_up_to_and_past_its_table(gpu_api, monkeypatch):
    """The dictionary built for a few distinct blocks has room for ``table_cap`` entries (three quarters of its initial
    2^16 hash table): a scatter that brings it just under stays a patch, the next one that passes it rebuilds."""
    lattice = gpu_api.CubicLattice((250, 250, 1))
    system = vc.fill(gpu_api, gpu_api.Hamiltonian(lattice), list(lattice.bonds()), "diag")
    sysn = system._sys
    vc.set_env(monkeypatch, ())
    stats, distinct = _begin_stats(sysn)
    hash_slots = 1 << 16   # dict_build's first hash table, kept while fewer than half of it is used
    assert 0 < distinct < hash_slots // 2
    table_cap = min(max(distinct + distinct // 2, distinct + 65536), hash_slots * 3 // 4)
    n_blocks = len(sysn.export_bsr(False)[1])
    σ0, σ3 = gpu_api.σ0, gpu_api.σ3

    def onsite(sites, first):
        return pc.packed(h=[(s, s, (2.0 + (first + k) * 2.0**-20) * σ0 - 0.05 * σ3) for k, s in enumerate(sites)])

    # (1) distinct new on-site blocks up to one entry below the capacity: patched
    first = table_cap - 1 - distinct
    assert first * 4 <= n_blocks
    system.fill(*onsite(range(first), 0))
    now, distinct = _begin_stats(sysn)
    assert now["patched_scatters"] == stats["patched_scatters"] + 1 and now["native_builds"] == stats["native_builds"], now
    assert distinct == table_cap - 1
    _check_copies(gpu_api, system, monkeypatch, True, (), 8, "below table_cap")

    # (2) ten more: the table is full, the copies are rebuilt
    stats = sysn.stats()
    system.fill(*onsite(range(first, first + 10), first))
    now, _ = _begin_stats(sysn)
    assert now["patched_scatters"] == stats["patched_scatters"], now
    assert now["native_builds"] == stats["native_builds"] + 1 and now["compactions"] == stats["compactions"] + 1, now
    H = system.matrix("bsr")
    scale = system.spectral_bound()
    want = orc.cheb_moments(H, orc.rademacher(SEED, H.shape[0], np.arange(8)), 16, scale)
    for kernel in ("auto", "dict_diag", "dict", "pair"):
        got = system.chebyshev_moments(16, vectors=8, seed=SEED, scale=scale, kernel=kernel)
        assert rel_err(got, want) <= 1e-10, kernel
