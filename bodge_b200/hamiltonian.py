"""``Hamiltonian``: the reference's tight-binding front end on top of the CUDA library.

Same public surface as ``bodge/hamiltonian.py:5-387`` of the reference -- the context manager
handing out ``H[i, j]`` / ``Δ[i, j]`` dicts, ``matrix()``, ``index()``, ``diagonalize()``,
``free_energy()``, ``ldos()`` -- but the matrix lives on the GPU: the skeleton, the scatter with
particle-hole/Hermitian fill, the Hermiticity check, the zero-block compaction and the
Chebyshev/KPM expansion behind ``free_energy(cuda=True)`` and ``ldos()`` all run in
``libbdg.so`` (``csrc/*.cu``) through the C ABI in ``include/bdg.h``.

There is no CPU assembly path: constructing a ``Hamiltonian`` without a CUDA device (or without
the built library) raises ``RuntimeError``.
"""

from __future__ import annotations

import os
import warnings

from . import _native, distributed, kpm
from .common import *
from .helpers import dwave, pwave, ssd, swave  # the reference exports them from bodge.hamiltonian (hamiltonian.py:390-531)
from .lattice import CubicLattice, Lattice


class AccuracyWarning(UserWarning):
    """A KPM observable was asked for (or capped at) fewer Chebyshev moments than its tolerance needs."""


class _DeviceData(np.ndarray):
    """Host snapshot of the device-resident ``data`` array that WRITES THROUGH: the reference hands out the live
    array (``system._data``, advertised by ``index()``'s docstring: ``system._data[k, ...] = v``), so item assignment
    on this view -- or on any slice of it -- uploads the edited snapshot to the GPU."""

    def __new__(cls, array, owner):
        obj = np.asarray(array).view(cls)
        obj._owner, obj._root = owner, obj
        return obj

    def __array_finalize__(self, obj):
        self._owner = getattr(obj, "_owner", None)
        self._root = getattr(obj, "_root", None)

    def __setitem__(self, key, value):
        super().__setitem__(key, value)
        if self._owner is not None and self._root is not None:
            self._owner._scale_cache = None
            self._owner._sys.import_data(np.asarray(self._root))


def _default_device() -> int:
    return int(os.environ.get("LOCAL_RANK", "0"))


def _pack_entries(lattice: Lattice, entries: dict):
    """``{(coord_i, coord_j): 2x2}`` -> flat ``i``, ``j`` (int64) and values ``[n, 2, 2]`` complex128.

    The reference resolves every key with two type-checked ``lattice[...]`` calls
    (bodge/hamiltonian.py:164); here the keys are converted in bulk and indexed vectorised.
    """
    n = len(entries)
    if n == 0:
        none = np.zeros(0, dtype=np.int64)
        return none, none.copy(), np.zeros((0, 2, 2), dtype=np.complex128)
    # Fast path: one C loop over the dict (csrc/pack_dict.c) when every entry has the plain form the reference's
    # own examples use -- integer coordinate tuples and 2x2 complex128 arrays.
    vals = np.empty((n, 2, 2), dtype=np.complex128)
    if type(lattice) is CubicLattice and lattice.size < 2**31:  # stock lattice: flat indices in the same loop
        i, j = np.empty(n, dtype=np.int32), np.empty(n, dtype=np.int32)
        if _native.pack_dict_cubic(entries, lattice.shape, i, j, vals) == n:
            return i, j, vals
    keys = np.empty((n, 2, 3), dtype=np.int64)
    if _native.pack_dict(entries, keys, vals) != n:
        try:
            keys = np.array(list(entries.keys()))
        except (ValueError, TypeError, OverflowError) as err:
            raise TypeError("Hamiltonian keys must be pairs of integer (x, y, z) coordinates") from err
        if keys.shape != (n, 2, 3) or keys.dtype.kind not in "iu":
            raise TypeError("Hamiltonian keys must be pairs of integer (x, y, z) coordinates")
        keys = keys.astype(np.int64)
        try:
            vals = np.array(list(entries.values()), dtype=np.complex128)
            if vals.shape != (n, 2, 2):
                raise ValueError
        except ValueError:
            # Mixed shapes: the reference assigns with numpy broadcasting (hamiltonian.py:107-118).
            vals = np.stack([np.broadcast_to(np.asarray(v, dtype=np.complex128), (2, 2)) for v in entries.values()])
    i = lattice.index_many(keys[:, 0, :])
    j = lattice.index_many(keys[:, 1, :])
    return i, j, vals


class Hamiltonian:
    """Tight-binding Bogoliubov-de Gennes Hamiltonian ``Lattice ⊗ Nambu ⊗ Spin`` (4N x 4N).

    Usage is unchanged from the reference::

        system = Hamiltonian(CubicLattice((100, 100, 1)))
        with system as (H, Δ):
            for i in lattice.sites():
                H[i, i] = -μ * σ0
                Δ[i, i] = -Δs * jσ2
            for i, j in lattice.bonds():
                H[i, j] = -t * σ0
        F = system.free_energy(0.1, cuda=True)

    Additions (all optional): ``fill()`` takes packed arrays instead of dicts for
    million-site systems, ``chebyshev_moments()`` exposes the KPM engine, ``ldos_map()``
    evaluates the LDOS at many sites at once, and the observables accept keyword-only KPM knobs.
    """

    @typecheck
    def __init__(self, lattice: Lattice, *, device: int | None = None):
        self.lattice: Lattice = lattice
        self.shape: Indices = (4 * lattice.size, 4 * lattice.size)
        self.device = _default_device() if device is None else device

        # Skeleton on the device (reference: hamiltonian.py:37-64).  Cubic lattices use the
        # analytic periodic stencil; any other Lattice goes through its own iterator once.
        stock = isinstance(lattice, CubicLattice) and all(
            getattr(type(lattice), m) is getattr(CubicLattice, m) for m in ("index", "sites", "bonds", "edges"))
        if stock:
            self._sys = _native.System.cubic(lattice.shape, self.device)
        else:
            pairs = [(lattice[ri], lattice[rj]) for ri, rj in lattice]
            pi = np.array([p[0] for p in pairs], dtype=np.int64)
            pj = np.array([p[1] for p in pairs], dtype=np.int64)
            self._sys = _native.System.generic(lattice.size, pi, pj, self.device)
        self._structure = None  # host copy of (indptr, indices) of the skeleton, fetched lazily
        self._scale_cache = None

    # ------------------------------------------------------------------------------------
    # context manager: collect dict entries, scatter them on exit
    # ------------------------------------------------------------------------------------
    @typecheck
    def __enter__(self) -> tuple[dict[Coords, Matrix], dict[Coords, Matrix]]:
        self._hopp = {}
        self._pair = {}
        return self._hopp, self._pair

    @typecheck
    def __exit__(self, exc_type, exc_val, exc_tb):
        """Transfer ``H``/``Δ`` to the device matrix, fill the hole sector from particle-hole and
        Hermitian symmetry, verify Hermiticity (reference: hamiltonian.py:91-126).  Like the
        reference this runs even if the ``with`` body raised, and a non-Hermitian result raises
        ``RuntimeError`` while leaving the matrix modified."""
        h_i, h_j, h_val = _pack_entries(self.lattice, self._hopp)
        p_i, p_j, p_val = _pack_entries(self.lattice, self._pair)
        self.fill(h_i, h_j, h_val, p_i, p_j, p_val)
        del self._hopp
        del self._pair

    def fill(self, h_i, h_j, h_val, p_i=(), p_j=(), p_val=(), *, check_hermitian: bool = True) -> float:
        """Bulk equivalent of one ``with`` block: flat site indices + ``[n,2,2]`` values.

        ``H[i,j]`` entries ``(h_i, h_j, h_val)`` and ``Δ[i,j]`` entries ``(p_i, p_j, p_val)``; keys must
        be unique within each list.  Returns ``max|M - M^†|``.
        """
        self._scale_cache = None
        return self._sys.scatter(h_i, h_j, h_val, p_i, p_j, np.asarray(p_val, dtype=np.complex128).reshape(-1, 2, 2),
                                 herm_tol=1e-6 if check_hermitian else -1.0)

    # ------------------------------------------------------------------------------------
    # matrix access
    # ------------------------------------------------------------------------------------
    def _bsr(self, eliminate_zeros: bool) -> BsrMatrix:
        indptr, indices, data = self._sys.export_bsr(eliminate_zeros)
        return BsrMatrix((data, indices, indptr), shape=self.shape, blocksize=(4, 4))

    @property
    def _matrix(self) -> BsrMatrix:
        """Snapshot of the full skeleton (unset blocks are zero), as the reference's ``_matrix``."""
        return self._bsr(eliminate_zeros=False)

    @property
    def _data(self) -> Matrix:
        return _DeviceData(self._sys.export_bsr(False)[2], self)

    @_data.setter
    def _data(self, value):
        self._scale_cache = None
        self._sys.import_data(value)

    @typecheck
    def matrix(self, format: str = "dense") -> SpMatrix | Matrix:
        """Export as ``"dense"`` (default), ``"bsr"``, ``"csr"`` or ``"csc"``; sparse formats have
        their zeros eliminated (reference: hamiltonian.py:128-155)."""
        match format:
            case "bsr":
                return self._bsr(eliminate_zeros=True)
            case "csr":
                indptr, indices, data = self._sys.export_csr(transpose=False)
                return CsrMatrix((data, indices, indptr), shape=self.shape)
            case "csc":
                indptr, indices, data = self._sys.export_csr(transpose=True)
                return CscMatrix((data, indices, indptr), shape=self.shape)
            case "dense":
                return np.asmatrix(self._sys.export_dense())
            case _:
                raise RuntimeError("Requested matrix format is not yet supported")

    @typecheck
    def index(self, row: Coord, col: Coord) -> Index:
        """Position of block ``(row, col)`` in the skeleton's ``data`` (hamiltonian.py:157-170)."""
        i, j = self.lattice[row], self.lattice[col]
        return Index(self._sys.lookup([i], [j])[0])

    # ------------------------------------------------------------------------------------
    # Chebyshev / KPM engine
    # ------------------------------------------------------------------------------------
    def spectral_bound(self, method: str = "norm", *, vectors: int = 4, seed: int = 99, check_steps: int = 128) -> float:
        """Scale ``a`` that puts the spectrum of ``H / a`` strictly inside [-1, 1].

        ``"norm"`` (default, used when an observable is called without ``scale=``): ``1.01 * ||H||_inf``,
        the max absolute row sum -- cheap, deterministic, never too small.

        ``"lanczos"`` (SURVEY 8f-4): a tighter ``a``, so that fewer moments give the same energy
        resolution (``N ∝ a``).  The Chebyshev recursion itself is the Krylov process: 32 moments of a
        few random vectors give 16 Lanczos steps through the modified Chebyshev algorithm
        (``kpm.jacobi_from_moments``), the largest Ritz value plus its residual estimates
        ``max|ε|``, and the candidate ``a`` is then VERIFIED on the GPU: ``check_steps`` recursion
        steps at that scale must stay bounded (``<T_n|T_n> <= <x|x>``), which fails exponentially
        fast if any eigenvalue lies outside [-a, a].  Never larger than the ``"norm"`` bound.
        """
        if self._scale_cache is None:
            self._scale_cache = 1.01 * self._sys.norm_inf()
        safe = self._scale_cache
        if method == "norm":
            return safe
        if method != "lanczos":
            raise ValueError(f"unknown spectral bound method '{method}'")
        if safe <= 0:
            return safe

        def estimate(scale):
            mu = self.chebyshev_moments(32, vectors=vectors, seed=seed, scale=scale)
            return max(kpm.spectral_radius_from_moments(mu[:, c], scale)[1] for c in range(mu.shape[1]))

        est = estimate(safe)
        if 1.1 * est < safe:  # a tighter scale conditions the moment -> Lanczos map better: refine once
            est = min(est, estimate(1.1 * est))
        candidate = 1.01 * est
        for _ in range(6):
            if candidate >= safe:
                return safe
            mu = self.chebyshev_moments(2 * check_steps + 2, vectors=vectors, seed=seed + 1, scale=candidate)
            even = mu[0::2]  # mu_2n = 2 <T_n|T_n> - mu_0: bounded by mu_0 iff no eigenvalue outside [-a, a]
            if np.all(np.isfinite(even)) and np.all(even <= even[0] * (1 + 1e-9)):
                return min(safe, 1.005 * candidate)  # the check resolves excursions beyond ~0.3 %
            candidate *= 1.03
        return safe

    def _probe_rows(self, sites) -> np.ndarray:
        rows = []
        for site in sites:
            base = 4 * self.lattice[tuple(int(v) for v in site)]
            rows.extend(range(base, base + 4))
        return np.array(rows, dtype=np.int64)

    def chebyshev_moments(self, moments: int, *, rows=None, vectors: int | None = None, seed: int = 1234,
                          scale: float | None = None, summed: bool = False, kernel: str = "auto",
                          batch: int | None = None, group="auto") -> Matrix:
        """Chebyshev moments ``mu[n, c] = <x_c| T_n(H/scale) |x_c>``, ``n < moments``.

        Start vectors are either unit vectors ``e_r`` for the scalar rows in ``rows`` (``4*site + α``),
        or ``vectors`` Rademacher columns derived from ``seed``.  With ``summed=True`` the result
        is ``sum_c mu[n, c]`` (shape ``[moments]``).  When ``torch.distributed`` is initialised
        the columns are split over the ranks (each holds a replica of the matrix) and combined
        with one all-reduce / all-gather; every rank gets the full result.

        ``kernel``: ``"auto"`` picks the fastest step kernel the matrix qualifies for (``include/bdg.h``): on 2-D
        lattices with a few distinct blocks two applications of ``H`` per launch on the even Chebyshev vectors
        (``"t2"``), else the block-dictionary / fixed-width / generic BSR single-step kernels (``"dict_diag"``,
        ``"dict"``, ``"ell"``, ``"dmma"``); ``"pair"`` is the literal three-term recursion two steps per launch,
        ``"fma"`` a scalar A/B reference.  All agree to rounding (tests: <= 1e-10 against the CPU oracle).
        """
        return self._columns(moments, lambda sysn, k: sysn.cheb_read(moments, k, summed=summed), summed,
                             rows=rows, vectors=vectors, seed=seed, scale=scale, kernel=kernel, batch=batch, group=group)

    def _columns(self, moments, read, summed, *, rows=None, vectors=None, seed=1234, scale=None, kernel="auto",
                 batch=None, group="auto", begin=None):
        """Run the recursion for ``moments`` moments over all start columns -- sharded over the
        ranks of the process group, in batches on this GPU -- and reduce each batch ON THE DEVICE
        with ``read(system, n_columns)``, which returns ``[m, n_columns]`` (per column) or ``[m]``
        (``summed``).  One collective combines the ranks.

        ``begin(system, c0, c1)`` is called after each batch's ``cheb_begin`` with the batch's columns ``[c0, c1)`` of
        the full list, to register a local accumulator.  ``moments`` is then the length of a series without moment
        doubling (``moments - 1`` steps), and ``kernel="auto"`` stays on kernels that keep every vector."""
        if (rows is None) == (vectors is None):
            raise ValueError("give either rows= (probe columns) or vectors= (random columns)")
        scale = self.spectral_bound() if scale is None else float(scale)
        n_total = len(rows) if rows is not None else int(vectors)
        rows = None if rows is None else np.asarray(rows, dtype=np.int64)
        rank, world, group = distributed.resolve(group)
        lo, hi = distributed.shard_range(n_total, rank, world)
        n_local = hi - lo
        if batch is None:  # two vector sets of 64*N*k bytes each (four with the pair kernel); keep two under ~16 GB
            batch = max(8, int(8e9 // (64 * self.lattice.size)) // 8 * 8)
        steps = (moments + 1) // 2 - 1 if begin is None else moments - 1
        if kernel == "auto" and begin is None:   # only moments are read here: the library may keep every second vector only
            kernel = "auto_moments"
        parts = []
        for b0 in range(0, n_local, batch):
            b1 = min(n_local, b0 + batch)
            if rows is not None:
                self._sys.cheb_begin(probe_rows=rows[lo + b0 : lo + b1], scale=scale, kernel=kernel)
            else:
                self._sys.cheb_begin(n_random=b1 - b0, seed=seed, col_offset=lo + b0, scale=scale, kernel=kernel)
            if begin is not None:
                begin(self._sys, lo + b0, lo + b1)
            done = self._sys.cheb_available() // 2 - 1      # steps bdg_cheb_begin has already taken (1 with T2)
            self._sys.cheb_steps(max(0, steps - done))
            parts.append(np.asarray(read(self._sys, b1 - b0), dtype=np.float64))
        if summed:
            local = np.sum(parts, axis=0) if parts else None
        else:
            local = np.concatenate(parts, axis=1) if parts else None
        if local is None:  # this rank got no columns: learn the leading dimension from a dry call shape
            m = self._leading_dim(read, moments)
            local = np.zeros(m) if summed else np.zeros((m, 0))
        return distributed.combine(local, summed, n_total, rank, world, group, device=self.device)

    @staticmethod
    def _leading_dim(read, moments):
        return getattr(read, "leading_dim", moments)

    # ------------------------------------------------------------------------------------
    # observables
    # ------------------------------------------------------------------------------------
    @typecheck
    def diagonalize(
        self, cuda: bool = False, format: str = "reshape"
    ) -> tuple[Matrix, Matrix] | dict[float, tuple[Matrix, Matrix, Matrix, Matrix]]:
        """Positive eigenvalues and their eigenvectors by dense diagonalisation
        (reference: hamiltonian.py:172-251).  Out of the hot path: delegated to LAPACK (scipy), or
        to cuSOLVER through torch when ``cuda=True``.  ``format="reshape"`` returns
        ``eigvec[n, site, α]``, ``format="raw"`` the column eigenvectors."""
        H = self.matrix(format="dense")
        if cuda:
            try:
                import torch
            except ModuleNotFoundError:
                raise RuntimeError("`cuda=True` needs torch with CUDA support for the dense eigensolver.")
            if not torch.cuda.is_available():
                raise RuntimeError("`cuda=True` needs a CUDA device.")
            dev = torch.device("cuda", self.device)
            _native.release_cached(self.device)  # the library's recycled buffers go back to the driver before torch allocates
            w, v = torch.linalg.eigh(torch.as_tensor(np.asarray(H), device=dev))
            eigval, eigvec = w.cpu().numpy(), v.cpu().numpy()
            keep = np.where(eigval > 0)
            eigval, eigvec = eigval[keep], eigvec[:, keep]
        else:
            eigval, eigvec = la.eigh(H, subset_by_value=(0.0, np.inf), overwrite_a=True, driver="evr")
            eigval, eigvec = np.array(eigval), np.array(eigvec)
        if format == "raw":
            return eigval, eigvec
        if format == "reshape":
            return eigval, eigvec.T.reshape((eigval.size, -1, 4))
        raise RuntimeError(f"Eigenstate format '{format}' is not yet supported.")

    @typecheck
    def free_energy(self, temperature: float = 0.0, cuda: bool = False, *, moments: int | None = None,
                    vectors: int | None = None, seed: int = 1234, scale: float | None = None,
                    kernel: str = "auto", tol: float = 1e-13) -> float:
        """Landau free energy ``F = U - TS`` of the BdG quasiparticles (hamiltonian.py:253-321).

        ``cuda=False``: the reference's algorithm, a dense ``eigvalsh`` (LAPACK through scipy) -- exact.

        ``cuda=True``: kernel-polynomial expansion on the GPU.  ``F = Tr g(H)`` with
        ``g(ε) = -(T/2) ln(1 + e^{-ε/T})`` is expanded in ``moments`` Chebyshev polynomials of
        ``H/scale``; the trace is exact (all 4N unit vectors) when ``vectors is None``, else a
        stochastic estimate from ``vectors`` Rademacher columns.  Accuracy of the expansion (the reference's
        ``cuda=True`` is an exact dense eigensolver, so this is the one place the two differ):

        * T > 0: the series converges like ``exp(-n π T / scale)``; ``moments=None`` picks the length for a relative
          truncation error ``tol`` (default 1e-13: 1e-12 agreement with the dense path measured at C1), capped at
          32768 terms -- below ``T ≈ 1e-3 · scale`` the cap bites and an ``AccuracyWarning`` states the level reached;
        * T = 0 (the API default): ``g`` has a kink at the Fermi level, the series converges only algebraically --
          about 1e-7 relative at the default 8192 moments, 1e-4 in the worst cases -- and an ``AccuracyWarning``
          says so; use ``cuda=False`` or a small finite T when more is needed;
        * an explicit ``moments`` below what ``tol`` asks for warns too;
        * sites nothing couples to (a geometry cut out of the lattice by leaving sites unset): their rows are zero, LAPACK
          returns their eigenvalues as exactly 0.0 and the reference's ``ε > 0`` filter (hamiltonian.py:304) drops them,
          while a trace counts ``g(0) = -(T/2) ln 2`` for each.  The zero rows are counted on the device and their share
          is taken out again, so the result is the reference's; a matrix that is identically zero returns 0 like it.

        Multi-GPU: columns are sharded over the initialised ``torch.distributed`` group.
        """
        T = temperature
        if T < 0:
            raise ValueError("Expected non-negative temperature!")
        if not cuda:
            ε = la.eigvalsh(self.matrix(format="dense"))
            ε = ε[ε > 0]
            S = np.sum(np.log(1 + np.exp(-ε / T))) if T > 0 else 0
            return float(-(1 / 2) * np.sum(ε) - T * S)

        scale = self.spectral_bound() if scale is None else float(scale)
        if scale == 0.0:
            # the matrix is identically zero (nothing set yet): no positive eigenvalue, the reference's sums over ε > 0
            # are empty (hamiltonian.py:302-319) -- and there is no interval to map onto [-1, 1]
            return 0.0
        need, reached = kpm.free_energy_moments(T, scale, tol)
        n_mom = need if moments is None else int(moments)
        if T == 0:
            warnings.warn("free_energy(cuda=True) at T = 0 expands the kinked g(ε) = min(ε, 0)/2 in Chebyshev polynomials: "
                          f"expect ~{reached * (need / max(n_mom, 1)) ** 2:.0e} relative error with {n_mom} moments (algebraic "
                          "convergence); cuda=False is exact, a small finite T converges geometrically", AccuracyWarning, stacklevel=2)
        elif n_mom < need or reached > tol:
            level = max(reached, kpm.series_error(n_mom, np.pi * T / scale))
            warnings.warn(f"free_energy(cuda=True): {n_mom} moments at T = {T:g}, scale = {scale:.3g} truncate the series at "
                          f"~{level:.1e} relative (tol = {tol:g} needs {int(np.ceil(-np.log(tol) * scale / (np.pi * T)))})",
                          AccuracyWarning, stacklevel=2)
        # F = sum_n c_n Tr T_n(H/scale): the series is contracted with the moments on the device,
        # so one double per GPU crosses PCIe / NVLink instead of the moment arrays.
        coef = kpm.chebyshev_coefficients(lambda e: kpm.free_energy_density(e, T), n_mom, scale)

        def read(sysn, k):
            return np.array([sysn.kpm_contract(coef, k, summed=True)])

        read.leading_dim = 1
        # what the all-zero rows add to a trace and the reference leaves out (see the docstring); g(0) = 0 at T = 0
        isolated = -0.5 * T * np.log(2.0) * self._sys.zero_scalar_rows() if T > 0 else 0.0
        if vectors is None:
            if self.shape[0] > (1 << 18):
                # the reference's exact path (dense eigvalsh) stops being possible long before this size; the exact KPM
                # trace still works but is O(N^2): say so instead of silently running for hours
                warnings.warn(f"free_energy(cuda=True) without vectors= takes the exact trace over all {self.shape[0]} unit "
                              "columns (O(N^2) work); pass vectors=64 or so for a stochastic estimate (relative error "
                              "~ 1/sqrt(vectors * 4N))", AccuracyWarning, stacklevel=2)
            total = self._columns(n_mom, read, True, rows=np.arange(self.shape[0]), scale=scale, kernel=kernel)
            return float(total[0] - isolated)
        total = self._columns(n_mom, read, True, vectors=vectors, seed=seed, scale=scale, kernel=kernel)
        return float(total[0] / vectors - isolated)   # (a Rademacher column has weight 1 on every row: the same share)

    @typecheck
    def ldos(self, site: Coord, energies: Matrix | list[float], *, moments: int | None = None,
             scale: float | None = None, kernel: str = "auto", tol: float = 1e-13) -> Matrix:
        """Local density of states at ``site`` (hamiltonian.py:323-387).

        Same definition as the reference -- ``ρ(±ε) = -Im Σ_σ [(ε + iΓ - H)^{-1}]_{σσ} / π`` with
        ``Γ = np.gradient(unique(|ε|))`` -- but the resolvent diagonal is evaluated from the
        Chebyshev moments of the four unit vectors at ``site`` (one GPU recursion for all
        energies) instead of one sparse LU solve per energy.  ``moments=None`` takes as many as the smallest
        broadening needs for a truncation error ``tol`` (``≈ 30·scale/Γ``); fewer -- passed explicitly, or because the
        2^20 cap bites -- raise an ``AccuracyWarning``: the truncated series oscillates and may turn negative where
        the reference's exact solve cannot."""
        return self.ldos_map([site], energies, moments=moments, scale=scale, kernel=kernel, tol=tol)[0]

    def ldos_map(self, sites, energies, *, moments: int | None = None, scale: float | None = None,
                 kernel: str = "auto", tol: float = 1e-13) -> Matrix:
        """LDOS at many sites: ``result[s, e]``; all ``4 * len(sites)`` probe columns run together
        (sharded over GPUs when ``torch.distributed`` is initialised)."""
        energies = np.array(energies, dtype=float)
        scale = self.spectral_bound() if scale is None else float(scale)
        eps = np.unique(np.abs(energies))
        if eps.size < 2:
            raise ValueError("need at least two distinct |energies| to define the broadening Γ")
        if scale == 0.0:
            # H = 0: every diagonal element of the resolvent is (ε + iΓ)^-1, what the reference's solve returns for it
            rows = self._probe_rows(sites)  # (coordinates are validated like on the normal path)
            g_imag = np.broadcast_to(np.imag(1.0 / (eps + 1j * np.gradient(eps))), (len(rows) // 4, 4, len(eps)))
            return kpm.ldos_from_resolvent(g_imag, eps, energies)
        gamma_min = float(np.min(np.abs(np.gradient(eps))))
        need, reached = kpm.ldos_moments(scale, gamma_min, tol)
        moments = need if moments is None else int(moments)
        if moments < need or reached > tol:
            # the reference's spsolve LDOS is exact and >= 0 by construction (tests/test_hamiltonian.py:498-500);
            # a truncated resolvent series oscillates around it and can dip below zero
            level = max(reached, kpm.series_error(moments, gamma_min / scale))
            warnings.warn(f"ldos: {moments} moments truncate the resolvent series at ~{level:.1e} of its leading term (broadening "
                          f"Γ = {gamma_min:.3g}, scale = {scale:.3g}: tol = {tol:g} needs {int(np.ceil(-np.log(tol) * scale / gamma_min))}); "
                          "the result may oscillate and turn negative", AccuracyWarning, stacklevel=3)
        # Resolvent diagonal at z = (ε + iΓ)/scale for every probe column and energy, evaluated on
        # the device from the moments (csrc/observables.cu); only [n_columns, n_energies] comes back.
        w, pref = kpm.resolvent_weights((eps + 1j * np.gradient(eps)) / scale)
        pref = pref / scale

        def read(sysn, k):
            g = sysn.kpm_resolvent(moments, k, w, pref)             # complex [k, n_eps]
            return np.concatenate([g.real.T, g.imag.T], axis=0)     # [2 n_eps, k]: columns last for the gather

        read.leading_dim = 2 * len(eps)
        out = self._columns(moments, read, False, rows=self._probe_rows(sites), scale=scale, kernel=kernel)
        g_imag = out[len(eps):].T.reshape(len(sites), 4, len(eps))  # Im G[site, α, ε]
        return kpm.ldos_from_resolvent(g_imag, eps, energies)

    # ------------------------------------------------------------------------------------
    # expectation values: local elements of the Fermi function f(H) (no reference code; the reference
    # would need diagonalize(), a dense O((4N)^3) eigensolver)
    # ------------------------------------------------------------------------------------
    def _flat(self, coords) -> np.ndarray:
        return np.array([self.lattice[tuple(int(v) for v in c)] for c in coords], dtype=np.int64)

    def _fermi_local(self, temperature, rows, read_col, read_site, *, moments=None, scale=None, tol=1e-13,
                     kernel="auto", batch=None, caller="density_matrix"):
        """``acc[r, α] = f(H)[4 read_site[r] + α, rows[read_col[r]]]`` as complex ``[n_reads, 4]``: one probe column
        per entry of ``rows``, the Fermi series contracted on the device while the recursion runs (``bdg.h``:
        ``bdg_cheb_local_begin``).  Columns are batched and sharded like every other observable; the reads of a batch
        land in their slots of one ``[n_reads, 4]`` array, so the ranks combine with a plain sum."""
        T = float(temperature)
        if not T > 0:
            raise ValueError(f"{caller} needs a temperature T > 0 (the Fermi function at T = 0 is a step function)")
        rows = np.asarray(rows, dtype=np.int64)
        read_col = np.asarray(read_col, dtype=np.int64)
        read_site = np.asarray(read_site, dtype=np.int64)
        n_reads = len(read_col)
        scale = self.spectral_bound() if scale is None else float(scale)
        if scale == 0.0:  # H = 0: f(H) = f(0) 1 = 1/2
            alpha = 4 * read_site[:, None] + np.arange(4)
            return np.where(alpha == rows[read_col][:, None], 0.5, 0.0).astype(np.complex128)
        need, reached = kpm.free_energy_moments(T, scale, tol)
        n_coef = need if moments is None else int(moments)
        if n_coef < need or reached > tol:
            level = max(reached, kpm.series_error(n_coef, np.pi * T / scale))
            warnings.warn(f"{caller}: {n_coef} moments at T = {T:g}, scale = {scale:.3g} truncate the Fermi series at "
                          f"~{level:.1e} relative (tol = {tol:g} needs {int(np.ceil(-np.log(tol) * scale / (np.pi * T)))})",
                          AccuracyWarning, stacklevel=3)
        coef = kpm.fermi_coefficients(T, n_coef, scale)
        batch_reads = []

        def begin(sysn, c0, c1):
            mine = np.flatnonzero((read_col >= c0) & (read_col < c1))
            batch_reads.append(mine)
            if len(mine):
                sysn.cheb_local_begin(coef, read_col[mine] - c0, read_site[mine])

        def read(sysn, k):
            full = np.zeros((n_reads, 4), dtype=np.complex128)
            mine = batch_reads[-1]
            if len(mine):
                full[mine] = sysn.cheb_local_read(len(mine))
            return full.view(np.float64).ravel()

        read.leading_dim = 8 * n_reads
        total = self._columns(n_coef, read, True, rows=rows, scale=scale, kernel=kernel, batch=batch, begin=begin)
        return np.ascontiguousarray(total, dtype=np.float64).view(np.complex128).reshape(n_reads, 4)

    def density_matrix(self, temperature: float, pairs, *, moments: int | None = None, scale: float | None = None,
                       tol: float = 1e-13, kernel: str = "auto", batch: int | None = None) -> Matrix:
        """Blocks of the one-body density matrix ``ρ = f(H)``, ``f(ε) = 1/(1 + e^{ε/T})``: complex
        ``[len(pairs), 4, 4]`` with ``result[p] = f(H)[4i:4i+4, 4j:4j+4]`` for ``pairs[p] = (i, j)`` (coordinates, like
        ``H[i, j]`` keys; basis e↑, e↓, h↑, h↓).  With the Nambu spinor ``Ψ = (c↑, c↓, c↑†, c↓†)``,
        ``<Ψ_a Ψ_b†> = δ_ab - ρ_ab``: e.g. ``<c_i↑ c_i↓> = -ρ[4i, 4i+3]``.

        A pair must be on-site or a block of the lattice's skeleton (``IndexError`` otherwise, like ``index()``);
        coordinates outside the lattice raise ``ValueError``.  The four scalar rows of every distinct ``j`` are probe
        columns of one Chebyshev recursion of ``f`` (no damping kernel: ``f`` is analytic for T > 0); the blocks are
        read at the requested ``i`` while it runs, on the GPU.  ``moments=None`` takes the series length for a relative
        truncation error ``tol``, the rule of ``free_energy`` (capped at 32768 terms); an explicit ``moments`` below
        that, or the cap, raise an ``AccuracyWarning``.  The series has no moment doubling: ``moments - 1`` steps.
        ``kernel="auto"`` runs the pair or a single-step kernel (the even-vector ``"t2"`` keeps every second vector
        only and is refused).  T <= 0 raises ``ValueError``."""
        pairs = list(pairs)
        i = self._flat([p[0] for p in pairs])
        j = self._flat([p[1] for p in pairs])
        off = i != j
        if off.any():
            self._sys.lookup(i[off], j[off])  # IndexError for a pair that is no block of the skeleton
        uj, pos = np.unique(j, return_inverse=True)
        rows = (4 * uj[:, None] + np.arange(4)).ravel()
        read_col = (4 * pos[:, None] + np.arange(4)).ravel()  # read 4p + β: column (j_p, β) at site i_p
        read_site = np.repeat(i, 4)
        acc = self._fermi_local(temperature, rows, read_col, read_site, moments=moments, scale=scale, tol=tol,
                                kernel=kernel, batch=batch, caller="density_matrix")
        return acc.reshape(len(pairs), 4, 4).transpose(0, 2, 1).copy()  # acc[4p + β, α] -> [p, α, β]

    def _potential(self, potential, sites):
        """``(coordinates, flat indices, V)`` of the sites an order parameter is asked for."""
        if isinstance(potential, dict):
            table = {int(k): float(v) for k, v in zip(self._flat(list(potential)), potential.values())}
        else:
            table = None
        if sites is None:
            sites = [s for s in self.lattice.sites()
                     if (table.get(self.lattice[s], 0.0) if table is not None else float(potential)) != 0.0]
        sites = [tuple(int(v) for v in s) for s in sites]
        flat = self._flat(sites)
        V = np.array([table.get(int(k), 0.0) for k in flat] if table is not None else np.full(len(flat), float(potential)))
        return sites, flat, V

    def order_parameter(self, temperature: float, potential, sites=None, **kpm_options) -> Matrix:
        """Mean-field s-wave order parameter ``Δ_i = -V_i ρ[4i, 4i+3]`` (complex, one per site) of an on-site attraction
        ``-V_i n_i↑ n_i↓``; ``Δ[i, i] = Δ_i jσ2`` is the pairing entry that reproduces it (``Δ[i, i] = -Δs jσ2`` is
        ``Δ_i = -Δs``).  It makes ``F + Σ_i |Δ_i|²/V_i`` stationary, with ``F`` from ``free_energy``.

        ``potential``: one ``V`` for every site, or a ``{site: V}`` dict; ``sites`` defaults to every site with
        ``V_i != 0``.  One probe column per site (row ``4i+3``) and one read, a quarter of ``density_matrix``'s work
        for the same sites.  ``kpm_options``: ``moments``, ``scale``, ``tol``, ``kernel``, ``batch`` as there."""
        sites, flat, V = self._potential(potential, sites)
        if len(flat) == 0:
            return np.zeros(0, dtype=np.complex128)
        acc = self._fermi_local(temperature, 4 * flat + 3, np.arange(len(flat)), flat, caller="order_parameter",
                                **kpm_options)
        return -V * acc[:, 0]

    def selfconsistent(self, temperature: float, potential, *, tol: float = 1e-8, max_iter: int = 500,
                       mixing: float = 1.0, **kpm_options) -> tuple[Matrix, int]:
        """Solve the s-wave gap equation ``Δ_i = -V_i ρ[4i, 4i+3]`` by plain fixed-point iteration: compute ``Δ``
        (``order_parameter``), write ``Δ[i, i] = Δ_i jσ2`` back (pairing entries only: the hopping stays), repeat until
        ``max_i |Δ_i^new - Δ_i| <= tol``.  ``mixing`` < 1 moves only that fraction of the way per iteration.  Starts
        from the pairing the system holds (set a non-zero guess: ``Δ = 0`` is always a fixed point) and leaves the
        last state in it.  Each iteration rewrites N of the ~5N blocks of a square lattice, which the library patches
        into its copies of the matrix in place.  Returns ``(Δ, iterations)``; warns if ``max_iter`` is reached."""
        if not 0 < mixing <= 1:
            raise ValueError("mixing must be in (0, 1]")
        sites, flat, V = self._potential(potential, None)
        if len(flat) == 0:
            return np.zeros(0, dtype=np.complex128), 0
        delta = self._sys.export_bsr(False)[2][self._sys.lookup(flat, flat), 0, 3]
        for it in range(1, int(max_iter) + 1):
            new = self.order_parameter(temperature, potential, sites, **kpm_options)
            step = np.max(np.abs(new - delta))
            delta = delta + mixing * (new - delta)
            self.fill((), (), (), flat, flat, delta[:, None, None] * jσ2)
            if step <= tol:
                return delta, it
        warnings.warn(f"selfconsistent: no convergence in {max_iter} iterations (last change {step:.2e} > tol = {tol:g})",
                      AccuracyWarning, stacklevel=2)
        return delta, int(max_iter)
