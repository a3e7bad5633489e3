"""Every Chebyshev step-kernel instantiation against an extended-precision reference (``variant_cases``).

For each ledger case the configuration is forced through the kernel name and the planner switches, and
``bdg_cheb_launched`` must list the instantiations the ledger assigns to it.  Then:

* (a) T_n and T_{n-1} after a few steps equal the ``np.clongdouble`` recursion over the exported BSR arrays to within
  ``K (n + 1) eps64 max(1, max|T|)`` -- a bound only rounding meets;
* (b) the per-column moments equal the oracle's to 1e-10 (norm-wise) and the summed moments their sum to 1e-13;
* (c) the vectors do not depend on the plan (row walk, patches, segments, classic or work-list plan), the pair kernel
  reproduces the single-step kernel of its format, the cube kernel the diagonal-hopping kernel, and a repeated run
  gives the same bits.

The local accumulator is checked against ``sum_n c_n T_n x`` of the same reference with random coefficients.
"""

import numpy as np
import pytest

import fermi_oracle as fo
import variant_cases as vc
from oracle import bdg_oracle as orc
from util import rel_err

pytestmark = pytest.mark.gpu
SEED = 11


@pytest.fixture(scope="module")
def systems(gpu_api):
    cache = {}

    def get(geometry, model):
        if (geometry, model) not in cache:
            system = vc.build(gpu_api, geometry, model)
            scale = system.spectral_bound()
            ref = vc.Reference(*system._sys.export_bsr(True), scale)
            cache[geometry, model] = (system, ref, system.matrix("bsr"), scale)
        return cache[geometry, model]

    return get


def run(system, scale, monkeypatch, case, env=None, kernel=None, steps=None):
    """One forced recursion: (launched short names, T_n index n, T_n, T_{n-1} or None, moments, summed moments)."""
    vc.set_env(monkeypatch, case.env if env is None else env)
    sysn = system._sys
    kernel = kernel or case.kernel
    sysn.cheb_begin(n_random=case.n_cols, seed=SEED, scale=scale, kernel=kernel)
    sysn.cheb_steps(case.steps if steps is None else steps)
    n = sysn.cheb_available() // 2
    launched = vc.short_names(sysn.cheb_launched())
    even_only = sysn.cheb_format()["kernel"] == "t2"
    cur = sysn.cheb_vectors(case.n_cols, 0)
    prev = None if even_only else sysn.cheb_vectors(case.n_cols, 1)
    mu = sysn.cheb_read(2 * n, case.n_cols)
    summed = sysn.cheb_read(2 * n, case.n_cols, summed=True)
    sysn.cheb_end()
    return launched, n, cur, prev, mu, summed


@pytest.mark.parametrize("case_id", sorted(vc.CASES))
def test_kernel_against_extended_precision(systems, monkeypatch, case_id):
    case = vc.CASES[case_id]
    system, ref, H, scale = systems(case.geometry, case.model)
    launched, n, cur, prev, mu, summed = run(system, scale, monkeypatch, case)
    assert set(case.kernels) <= set(launched), f"launched {launched}, the ledger expects {case.kernels}"

    x0 = orc.rademacher(SEED, H.shape[0], np.arange(case.n_cols))
    want = ref.vectors(x0, n)
    ratio = vc.rounding_ratio(cur, want[n], n)
    assert ratio <= vc.K_ROUNDING, f"T_{n}: error {ratio:.1f} x (n+1) eps max|T| (bound {vc.K_ROUNDING})"
    if prev is not None:
        ratio = vc.rounding_ratio(prev, want[n - 1], n - 1)
        assert ratio <= vc.K_ROUNDING, f"T_{n - 1}: error {ratio:.1f} x n eps max|T| (bound {vc.K_ROUNDING})"

    assert rel_err(mu, orc.cheb_moments(H, x0, 2 * n, scale)) <= 1e-10
    assert rel_err(summed, mu.sum(axis=1)) <= 1e-13

    again = run(system, scale, monkeypatch, case)
    assert again[0] == launched
    assert np.array_equal(again[2], cur) and np.array_equal(again[4], mu) and np.array_equal(again[5], summed)


# ---- (c) plan invariance --------------------------------------------------------------------------------------------
ELL_PLANS = [(("BDG_ELL_WALK", 0),), (("BDG_ELL_PZ", 1),), (("BDG_ELL_PZ", 4), ("BDG_ELL_SEG", 3)), (("BDG_ELL_SEG", 1),),
             (("BDG_ELL_PREFETCH", 0),), (("BDG_ELL_PREFETCH", 2), ("BDG_ELL_SEG", 5))]
ELL_CASES = sorted(i for i, c in vc.CASES.items() if c.kernel in ("ell", "dict", "dict_diag") and c.geometry in ("square", "slab", "cube")
                   and c.n_cols >= 5)


@pytest.mark.parametrize("case_id", ELL_CASES)
def test_row_walk_does_not_change_the_vectors(systems, monkeypatch, case_id):
    case = vc.CASES[case_id]
    system, _, _, scale = systems(case.geometry, case.model)
    base = run(system, scale, monkeypatch, case)
    for plan in ELL_PLANS:
        got = run(system, scale, monkeypatch, case, env=case.env + plan)
        assert got[0] == base[0], plan
        assert np.array_equal(got[2], base[2]) and np.array_equal(got[3], base[3]), plan


PAIR_CASES = sorted(i for i, c in vc.CASES.items() if c.kernels[0].startswith("cheb_pair_step"))


def _flip(env, name):
    d = dict(env)
    return tuple((k, v) for k, v in env if k != name) + ((name, "0" if d.get(name) == "1" else "1"),)


@pytest.mark.parametrize("case_id", PAIR_CASES)
def test_pair_plans_and_single_step_agree(systems, monkeypatch, case_id):
    case = vc.CASES[case_id]
    system, _, _, scale = systems(case.geometry, case.model)
    base = run(system, scale, monkeypatch, case)
    plans = [_flip(case.env, "BDG_PAIR_BALANCE"),
             case.env + (("BDG_PAIR_P", 5), ("BDG_PAIR_SEG", 3)),
             _flip(case.env, "BDG_PAIR_BALANCE") + (("BDG_PAIR_P", 3), ("BDG_PAIR_SEG", 1)),
             case.env + (("BDG_PAIR_P", 14), ("BDG_PAIR_SEG", 5)),
             case.env + (("BDG_PAIR_OPEN", 0),)]
    for plan in plans:
        got = run(system, scale, monkeypatch, case, env=plan)
        assert np.array_equal(got[2], base[2]), plan
        if base[3] is not None:
            assert np.array_equal(got[3], base[3]), plan
    if case.kernel != "pair":
        return
    single = "dict_diag" if case.model == "diag" else "dict"
    want = run(system, scale, monkeypatch, case, kernel=single)
    assert not any(k.startswith("cheb_pair_step") for k in want[0])
    if case.geometry == "pair_torus":   # wrap-around neighbours are added in stencil order, not block-column order
        bound = 1e-13 * max(np.max(np.abs(want[2])), 1.0)
        assert np.max(np.abs(base[2] - want[2])) <= bound and np.max(np.abs(base[3] - want[3])) <= bound
    else:
        assert np.array_equal(base[2], want[2]) and np.array_equal(base[3], want[3])


CUBE_CASES = sorted(i for i, c in vc.CASES.items() if c.kernels[0].startswith("cheb_cube_step"))


@pytest.mark.parametrize("case_id", CUBE_CASES)
def test_cube_plans_agree_with_the_diagonal_kernel(systems, monkeypatch, case_id):
    case = vc.CASES[case_id]
    system, _, _, scale = systems(case.geometry, case.model)
    base = run(system, scale, monkeypatch, case)
    for seg in (2, 5):
        got = run(system, scale, monkeypatch, case, env=case.env + (("BDG_CUBE_SEG", seg),))
        assert got[0] == base[0] and np.array_equal(got[2], base[2]), seg
    got = run(system, scale, monkeypatch, case, env=_flip(case.env, "BDG_CUBE_BALANCE"))
    assert np.array_equal(got[2], base[2])
    want = run(system, scale, monkeypatch, case, kernel="dict_diag", steps=case.steps + 1)   # T_n with the same n
    assert want[1] == base[1]
    assert np.max(np.abs(base[2] - want[2])) <= 1e-13 * max(np.max(np.abs(want[2])), 1.0)


def test_plan_switches_hold_for_the_recursion(systems, monkeypatch):
    """cheb_begin reads the plan switches once: BDG_ELL_SD=0 set after it leaves the running recursion on the kernel
    with the real-diagonal on-site product, and the vectors are those of an undisturbed run."""
    case = vc.CASES["dict-square-gen-c13"]
    system, _, _, scale = systems(case.geometry, case.model)
    want = run(system, scale, monkeypatch, case)
    vc.set_env(monkeypatch, case.env)
    sysn = system._sys
    sysn.cheb_begin(n_random=case.n_cols, seed=SEED, scale=scale, kernel=case.kernel)
    monkeypatch.setenv("BDG_ELL_SD", "0")
    sysn.cheb_steps(case.steps)
    launched = vc.short_names(sysn.cheb_launched())
    cur, prev = sysn.cheb_vectors(case.n_cols, 0), sysn.cheb_vectors(case.n_cols, 1)
    sysn.cheb_end()
    assert launched == list(case.kernels) == want[0]
    assert np.array_equal(cur, want[2]) and np.array_equal(prev, want[3])


# ---- local accumulator ----------------------------------------------------------------------------------------------
LOCAL_RUNS = [  # (kernel, columns, environment, kernel that must run)
    ("dict_diag", 1, (), "cheb_step_ell<1, 5, 1, true, true, false>"),
    ("dict_diag", 2, (), "cheb_step_ell<2, 5, 1, true, true, false>"),
    ("dict_diag", 3, (), "cheb_step_ell<4, 5, 1, true, true, false>"),
    ("dict_diag", 13, (), "cheb_step_ell<8, 5, 1, true, true, false>"),
    ("pair", 13, (("BDG_PAIR_BALANCE", 0),), "cheb_pair_step<true, false, 0, false, false>"),
    ("pair", 41, (("BDG_PAIR_BALANCE", 1),), "cheb_pair_step<true, false, 0, false, true>"),
]
CHUNKS = (0, 1, 3, 2, 4)   # steps requested per call: uneven, and past the end of every series below


@pytest.mark.parametrize("n_coef", range(1, 8))
@pytest.mark.parametrize("kernel,n_cols,env,expect", LOCAL_RUNS, ids=[f"{k}-c{c}" for k, c, _, _ in LOCAL_RUNS])
def test_local_accumulator_against_extended_precision(systems, monkeypatch, kernel, n_cols, env, expect, n_coef):
    system, ref, H, scale = systems("pair_open", "diag")
    rng = np.random.default_rng(100 * n_cols + n_coef)
    coef = rng.uniform(-1.0, 1.0, n_coef)
    n_sites = H.shape[0] // 4
    # more than 32 reads (several CTAs of the accumulator), the ragged last panel, a duplicate read
    cols = np.concatenate([rng.integers(0, n_cols, 40), [n_cols - 1, n_cols - 1]])
    sites = np.concatenate([rng.integers(0, n_sites, 40), [n_sites - 1, n_sites - 1]])
    cols, sites = np.append(cols, cols[0]), np.append(sites, sites[0])
    vc.set_env(monkeypatch, env)
    sysn = system._sys
    sysn.cheb_begin(n_random=n_cols, seed=SEED, scale=scale, kernel=kernel)
    sysn.cheb_local_begin(coef, cols, sites)
    x0 = orc.rademacher(SEED, H.shape[0], np.arange(n_cols))
    T = ref.vectors(x0, sum(CHUNKS) + 1)
    rows = 4 * sites[:, None] + np.arange(4)
    t_max = max(1.0, max(float(np.max(np.abs(t))) for t in T[:n_coef]))
    done = 1   # T_0 and T_1 are added by cheb_local_begin
    for chunk in CHUNKS:
        sysn.cheb_steps(chunk)
        done += chunk
        got = sysn.cheb_local_read(len(cols))
        terms = min(done, n_coef - 1)
        want = sum(coef[k] * T[k][rows, cols[:, None]] for k in range(terms + 1))
        bound = (terms + 1) * np.finfo(np.float64).eps * t_max * np.sum(np.abs(coef))
        ratio = float(np.max(np.abs(got.astype(np.clongdouble) - want))) / bound
        assert ratio <= vc.K_ROUNDING, f"after T_{done}: error {ratio:.1f} x the rounding bound"
    assert np.array_equal(got[-1], got[0])
    assert expect in vc.short_names(sysn.cheb_launched())
    import torch

    dev = torch.zeros((len(cols), 4), dtype=torch.complex128, device=f"cuda:{system.device}")
    sysn.cheb_local_read(len(cols), device_ptr=dev.data_ptr())
    torch.cuda.synchronize(system.device)
    assert np.array_equal(dev.cpu().numpy(), got)
    sysn.cheb_end()


def test_order_parameter_on_a_balanced_plan(gpu_api, monkeypatch):
    system = vc.build(gpu_api, "pair_open", "diag")
    rho = fo.fermi_dense(system.matrix("dense"), 0.1)
    lat = system.lattice
    sites = [(x, y, 0) for x in range(12) for y in range(20)]
    want = np.array([-1.5 * rho[4 * lat[s], 4 * lat[s] + 3] for s in sites])
    vc.set_env(monkeypatch, (("BDG_PAIR_BALANCE", 1),))
    assert np.max(np.abs(system.order_parameter(0.1, 1.5, sites) - want)) <= 1e-10
