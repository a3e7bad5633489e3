"""Every Chebyshev step-kernel instantiation of ``libbdg.so`` and the case that reaches it, plus the extended-precision
reference the cases are checked against.

``CASES`` names one forced configuration per entry (model, lattice, kernel, columns, environment switches) and the
instantiations it must launch; ``LEDGER`` inverts it.  ``test_kernel_ledger.py`` checks that the ledger covers exactly
the recursion kernels built into the library, ``test_gpu_variants.py`` runs every case and confirms through
``bdg_cheb_launched`` that it launched what the ledger says.

Kernel names are compared in a short form, ``cheb_step_ell<8, 5, 1, true, false, false>``: the mangled names carry an
anonymous-namespace tag that differs from build to build.
"""

from __future__ import annotations

import re
import shutil
import subprocess
from dataclasses import dataclass, field

import numpy as np

FAMILIES = ("cheb_step_ell", "cheb_step_dmma", "cheb_step_fma", "cheb_pair_step", "cheb_cube_step")
_SHORT = re.compile(r"(cheb_[a-z_]+<[^<>]*>)")


def short_names(names) -> list[str]:
    """``cheb_xxx<args>`` of mangled (``_Z...``) or demangled kernel names; names of other kernels are dropped."""
    names = list(names)
    mangled = [n for n in names if n.startswith("_Z")]
    if mangled:
        tool = shutil.which("c++filt") or shutil.which("cu++filt")
        if tool is None:
            raise RuntimeError("c++filt is needed to demangle kernel names")
        out = subprocess.run([tool], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout.split("\n")
        plain = dict(zip(mangled, out))
        names = [plain.get(n, n) for n in names]
    short = []
    for n in names:
        m = _SHORT.search(n)
        if m and m.group(1).split("<")[0] in FAMILIES:
            short.append(m.group(1))
    return short


# ---- extended-precision reference ---------------------------------------------------------------------------------
def longdouble_check():
    assert np.finfo(np.longdouble).eps < 1e-18, "np.longdouble is no wider than float64 here: the reference would be weak"


class Reference:
    """The recursion ``T_0 = x``, ``T_1 = (1/s) H x``, ``T_{n+1} = (2/s) H T_n - T_{n-1}`` in ``np.clongdouble`` over the
    exported BSR arrays, with the float64 step factors the library passes to its kernels."""

    def __init__(self, indptr, indices, data, scale):
        longdouble_check()
        self.n = len(indptr) - 1
        counts = np.diff(indptr)
        assert (counts > 0).all(), "every block row needs a block (reduceat)"
        self.starts = np.asarray(indptr[:-1], dtype=np.int64)
        self.indices = np.asarray(indices, dtype=np.int64)
        self.data = np.asarray(data).astype(np.clongdouble)
        self.a1 = np.longdouble(1.0 / scale)
        self.a2 = np.longdouble(2.0 / scale)

    def matvec(self, x):
        c = x.shape[1]
        xs = x.reshape(self.n, 4, c)[self.indices]
        prod = np.matmul(self.data, xs)
        return np.add.reduceat(prod, self.starts, axis=0).reshape(4 * self.n, c)

    def vectors(self, x0, n):
        """``[T_0, ..., T_n]`` of the start columns ``x0`` (``[4N, C]``)."""
        out = [np.asarray(x0).astype(np.clongdouble)]
        if n >= 1:
            out.append(self.a1 * self.matvec(out[0]))
        for _ in range(2, n + 1):
            out.append(self.a2 * self.matvec(out[-1]) - out[-2])
        return out


K_ROUNDING = 64


def rounding_ratio(got, want, n):
    """``max|got - want| / ((n + 1) eps64 max(1, max|want|))``: must stay <= K_ROUNDING for T_n."""
    want = np.asarray(want)
    err = float(np.max(np.abs(np.asarray(got).astype(np.clongdouble) - want)))
    scale = (n + 1) * np.finfo(np.float64).eps * max(1.0, float(np.max(np.abs(want))))
    return err / scale


# ---- models -------------------------------------------------------------------------------------------------------
def _pool(api, rng, n=3):
    return [-1.0 * api.σ0 + 0.3 * (rng.random((2, 2)) - 0.5 + 1j * (rng.random((2, 2)) - 0.5)) for _ in range(n)]


def fill(api, system, pairs, model, seed=7):
    """``model``: "diag" = README s-wave (on-site pairing, hopping -σ0: real-diagonal off-site blocks);
    "gen" = normal state with complex hopping from a pool of three 2x2 matrices and real-diagonal on-site blocks
    (dictionary with general off-site blocks, SD-eligible); "pairgen" = "gen" plus on-site pairing (not SD-eligible);
    "normal" = normal metal, hopping -σ0 and no pairing (real-diagonal off-site and on-site blocks: DIAG- and SD-eligible)."""
    rng = np.random.default_rng(seed)
    pool = _pool(api, rng)
    lattice = system.lattice
    with system as (H, D):
        for i in lattice.sites():
            H[i, i] = 3.0 * api.σ0 - 0.05 * api.σ3
            if model in ("diag", "pairgen"):
                D[i, i] = -0.2 * api.jσ2
        done = set()
        for i, j in pairs:
            if (i, j) in done or i == j:
                continue
            h = -1.0 * api.σ0 if model in ("diag", "normal") else pool[int(rng.integers(len(pool)))]
            H[i, j] = h
            H[j, i] = h.conj().T
            done.update(((i, j), (j, i)))
    return system


def hub_lattice(n_sites, degree):
    """A generic (non-cubic) lattice: an open chain ``0 - 1 - ... - n-1`` plus bonds from site 0 to sites 2 .. degree,
    so that row 0 holds ``degree + 1`` blocks."""
    from bodge_b200.lattice import Lattice

    class Hub(Lattice):
        def index(self, coord):
            if not (0 <= coord[0] < n_sites and coord[1] == 0 and coord[2] == 0):
                raise ValueError(f"Coordinate {coord} out of bounds")
            return coord[0]

        def sites(self):
            return iter([(i, 0, 0) for i in range(n_sites)])

        def bonds(self):
            out = []
            for i in range(n_sites - 1):
                out += [((i, 0, 0), (i + 1, 0, 0)), ((i + 1, 0, 0), (i, 0, 0))]
            for k in range(2, degree + 1):
                out += [((0, 0, 0), (k, 0, 0)), ((k, 0, 0), (0, 0, 0))]
            return iter(out)

        def edges(self):
            return iter([])

    return Hub((n_sites, 1, 1))


def periodic_pairs(lattice, x=True, y=True):
    in_plane = 1 if lattice.shape[2] == 1 else 2
    pairs = list(lattice.bonds())
    if x:
        pairs += list(lattice.edges(axis=0))
    if y:
        pairs += list(lattice.edges(axis=in_plane))
    return pairs


# geometry tag -> (lattice factory, pairs factory); the comment is the longest block row (ELL width)
GEOMETRIES = {
    "chain": lambda: ("cubic", (40, 1, 1)),        # 3
    "ladder": lambda: ("cubic", (20, 2, 1)),       # 4
    "square": lambda: ("cubic", (9, 17, 1)),       # 5; Ly Lz >= 16, Lx >= 8: the marching row walk applies
    "slab": lambda: ("cubic", (9, 8, 2)),          # 6; marching walk
    "cube": lambda: ("cubic", (8, 4, 5)),          # 7; marching walk
    "hub8": lambda: ("hub", (30, 7)),              # 8: one site bonded to 7 others
    "hub41": lambda: ("hub", (60, 40)),            # 41 blocks: DMMA tail loop past the one-lane-per-block index prefetch
    "pair_open": lambda: ("cubic", (12, 20, 1)),   # pair kernel: two patches of <= 14 sites per plane
    "pair_torus": lambda: ("torus", (11, 17, 1)),
    "cube3d": lambda: ("cubic", (6, 10, 11)),      # cube kernel: odd Lz, ragged patches for every shape
}
WIDTH = {"chain": 3, "ladder": 4, "square": 5, "slab": 6, "cube": 7, "hub8": 8}


def lattice_pairs(api, geometry):
    """The geometry's lattice and the (i, j) coordinate pairs its hopping is set on."""
    kind, arg = GEOMETRIES[geometry]()
    if kind == "hub":
        lattice = hub_lattice(*arg)
        return lattice, list(lattice.bonds())
    lattice = api.CubicLattice(arg)
    return lattice, periodic_pairs(lattice) if kind == "torus" else list(lattice.bonds())


def build(api, geometry, model):
    lattice, pairs = lattice_pairs(api, geometry)
    return fill(api, api.Hamiltonian(lattice), pairs, model)


# ---- planner switches ---------------------------------------------------------------------------------------------
PLAN_VARS = ("BDG_ELL_WALK", "BDG_ELL_PZ", "BDG_ELL_SEG", "BDG_ELL_PREFETCH", "BDG_ELL_SD", "BDG_PAIR_SELF", "BDG_PAIR_BALANCE",
             "BDG_PAIR_OPEN", "BDG_PAIR_P", "BDG_PAIR_SEG", "BDG_CUBE_SHAPE", "BDG_CUBE_BALANCE", "BDG_CUBE_SEG", "BDG_AUTO_PAIR",
             "BDG_AUTO_CUBE")


def set_env(monkeypatch, env):
    """Clear every planner switch, then set ``env`` (``((name, value), ...)``)."""
    for name in PLAN_VARS:
        monkeypatch.delenv(name, raising=False)
    for name, value in env:
        monkeypatch.setenv(name, str(value))


# ---- cases --------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    geometry: str
    model: str
    kernel: str
    n_cols: int
    env: tuple = ()                  # ((name, value), ...)
    steps: int = 6                   # cheb_steps after cheb_begin
    kernels: tuple = field(default=())  # instantiations it must launch (short names)

    @property
    def id(self):
        env = "".join(f"-{k[4:].lower()}{v}" for k, v in self.env)
        return f"{self.kernel}-{self.geometry}-{self.model}-c{self.n_cols}{env}"


def _pw(n_cols):
    return 8 if n_cols >= 5 else 4 if n_cols >= 3 else n_cols


def _b(v):
    return "true" if v else "false"


def _cases():
    out = []
    # single-step fixed-width kernels: cheb_step_ell<PW, CH, NP, DICT, DIAG, SD>
    for geo, width in WIDTH.items():
        for n_cols in (1, 2, 3, 13):
            pw = _pw(n_cols)
            out.append(Case(geo, "diag", "dict_diag", n_cols, kernels=(f"cheb_step_ell<{pw}, {width}, 1, true, true, false>",)))
            out.append(Case(geo, "gen", "dict", n_cols, kernels=(f"cheb_step_ell<{pw}, {width}, 1, true, false, true>",)))
            out.append(Case(geo, "gen", "dict", n_cols, env=(("BDG_ELL_SD", "0"),),
                            kernels=(f"cheb_step_ell<{pw}, {width}, 1, true, false, false>",)))
            # plain format: 13 columns on rows of >= 6 blocks take two panels per pass, one 8-column panel does not
            ell_cols = 7 if n_cols == 13 and width >= 6 else n_cols
            out.append(Case(geo, "gen", "ell", ell_cols, kernels=(f"cheb_step_ell<{_pw(ell_cols)}, {width}, 1, false, false, false>",)))
        if width >= 6:
            out.append(Case(geo, "gen", "ell", 13, kernels=(f"cheb_step_ell<8, {width}, 2, false, false, false>",)))
    # generic block rows: cheb_step_dmma<PW, FIRST, CH>, CH from the longest row; cheb_step_fma<PW, FIRST>
    for geo, ch in (("chain", 3), ("square", 5), ("cube", 7), ("hub41", 8)):
        for n_cols in (1, 2, 3, 13):
            pw = _pw(n_cols)
            out.append(Case(geo, "gen", "dmma", n_cols,
                            kernels=tuple(f"cheb_step_dmma<{pw}, {_b(first)}, {ch}>" for first in (True, False))))
    for n_cols in (1, 2, 3, 13):
        pw = _pw(n_cols)
        out.append(Case("hub41", "gen", "fma", n_cols, kernels=tuple(f"cheb_step_fma<{pw}, {_b(first)}>" for first in (True, False))))
    # two-steps-per-pass kernel: cheb_pair_step<DIAG, SELF, MODE, SD, LISTED>; 41 columns = six panels, the last ragged
    for model, diag, sd_env, sd in (("diag", True, (), False), ("gen", False, (), True), ("gen", False, (("BDG_ELL_SD", "0"),), False)):
        for self_ in (0, 1):
            for mode, kernel in ((0, "pair"), (1, "t2")):
                for listed in (0, 1):
                    geo = "pair_open" if listed == self_ else "pair_torus"
                    env = sd_env + (("BDG_PAIR_SELF", str(self_)), ("BDG_PAIR_BALANCE", str(listed)))
                    out.append(Case(geo, model, kernel, 41, env=env,
                                    kernels=(f"cheb_pair_step<{_b(diag)}, {_b(self_)}, {mode}, {_b(sd)}, {_b(listed)}>",)))
    # three-dimensional even-vector kernel: cheb_cube_step<16, PY, PZ, NE, LISTED>
    for shape, (py, pz, ne) in enumerate(((8, 8, 4), (6, 8, 5), (4, 8, 6))):
        for listed in (0, 1):
            n_cols = 37 if listed else 13
            out.append(Case("cube3d", "diag", "t2", n_cols, env=(("BDG_CUBE_SHAPE", str(shape)), ("BDG_CUBE_BALANCE", str(listed))),
                            kernels=(f"cheb_cube_step<16, {py}, {pz}, {ne}, {_b(listed)}>",)))
    return out


CASES = {c.id: c for c in _cases()}
assert len(CASES) == len(_cases()), "case ids must be unique"

LEDGER = {}
for _c in CASES.values():
    for _k in _c.kernels:
        assert _k not in LEDGER, f"{_k} is assigned to two cases"
        LEDGER[_k] = _c.id
