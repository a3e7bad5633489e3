"""ctypes binding of ``libbdg.so`` -- the thin layer between the Python surface and the C ABI
declared in ``include/bdg.h``.

No fallback: if the library is missing or no CUDA device is usable, the calls raise.  Return
codes are mapped to the exception types the reference raises in the same situation
(``bodge/hamiltonian.py:122,170``, ``bodge/lattice.py:106``).
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BDG_LIB") or os.path.join(_PKG, "libbdg.so")  # BDG_LIB: a development build of kernel variants

OK, E_INVALID, E_CUDA, E_NOT_NEIGHBOUR, E_NOT_HERMITIAN, E_OUT_OF_BOUNDS, E_NO_DEVICE = range(7)
X0_PROBE, X0_RADEMACHER = 0, 1
MU_PER_COLUMN, MU_SUM = 0, 1
KERNEL_AUTO, KERNEL_DMMA, KERNEL_FMA = 0, 1, 2
KERNELS = {"auto": KERNEL_AUTO, "dmma": KERNEL_DMMA, "fma": KERNEL_FMA, "ell": 3, "dict": 6, "dict_diag": 7, "pair": 8, "t2": 9,
           "auto_moments": 10}
KERNEL_NAMES = {v: k for k, v in KERNELS.items()}

_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_f64p = C.POINTER(C.c_double)
_vp = C.c_void_p

# name -> argument types (every function returns int unless noted); mirrors include/bdg.h.
SIGNATURES = {
    "bdg_abi_version": [],
    "bdg_device_count": [C.POINTER(C.c_int)],
    "bdg_destroy": [_vp],
    "bdg_release_cached": [C.c_int],
    "bdg_set_stream": [_vp, _vp],
    "bdg_sync": [_vp],
    "bdg_device_bytes": [_vp, _i64p],
    "bdg_pinned_alloc": [C.c_int64, C.POINTER(_vp)],
    "bdg_pinned_free": [_vp],
    "bdg_create_cubic": [C.c_int, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_vp)],
    "bdg_create_generic": [C.c_int, C.c_int64, C.c_int64, _vp, _vp, C.POINTER(_vp)],
    "bdg_skeleton_sizes": [_vp, _i64p, _i64p],
    "bdg_lookup": [_vp, C.c_int64, _vp, _vp, _vp, _i64p],
    "bdg_scatter": [_vp, C.c_int64, _vp, _vp, _vp, C.c_int64, _vp, _vp, _vp, C.c_double, _f64p, _i64p],
    "bdg_clear": [_vp],
    "bdg_stats": [_vp, _i64p],
    "bdg_export_bsr": [_vp, C.c_int, _i64p, _vp, _vp, _vp],
    "bdg_export_csr": [_vp, C.c_int, _i64p, _vp, _vp, _vp],
    "bdg_export_dense": [_vp, _vp],
    "bdg_import_data": [_vp, _vp],
    "bdg_norm_inf": [_vp, _f64p],
    "bdg_cheb_begin": [_vp, C.c_int, C.c_int32, _vp, C.c_uint64, C.c_int64, C.c_double, C.c_int],
    "bdg_cheb_steps": [_vp, C.c_int32, C.POINTER(C.c_float)],
    "bdg_cheb_reserve": [_vp, C.c_int32],
    "bdg_cheb_available": [_vp, C.POINTER(C.c_int32)],
    "bdg_cheb_moments_read": [_vp, C.c_int32, C.c_int, _vp, C.c_int],
    "bdg_cheb_moments": [_vp, C.c_int, C.c_int32, _vp, C.c_uint64, C.c_int64, C.c_double, C.c_int32, C.c_int, _vp, C.c_int],
    "bdg_cheb_moments_multi": [C.POINTER(_vp), C.c_int, C.c_int, C.c_int64, _vp, C.c_uint64, C.c_double, C.c_int32, C.c_int, _vp],
    "bdg_multi_release": [],
    "bdg_cheb_vectors": [_vp, C.c_int, _vp],
    "bdg_cheb_info": [_vp, _i64p, _i64p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), _i64p],
    "bdg_cheb_format": [_vp, C.POINTER(C.c_int32), _i64p, _i64p],
    "bdg_cheb_launched": [_vp, C.c_char_p, C.c_int64, _i64p],
    "bdg_cheb_end": [_vp],
    "bdg_kpm_resolvent": [_vp, C.c_int32, C.c_int32, _vp, _vp, _vp, C.c_int],
    "bdg_kpm_contract": [_vp, C.c_int32, _vp, C.c_int, _vp, C.c_int],
    "bdg_cheb_local_begin": [_vp, C.c_int32, _vp, C.c_int64, _vp, _vp],
    "bdg_cheb_local_read": [_vp, _vp, C.c_int],
}

_lib = None


def load():
    """Load ``libbdg.so`` (once).  Raises ``RuntimeError`` if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m bodge_b200.build` "
            "(bodge_b200 has no CPU fallback)"
        )
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    lib.bdg_last_error.argtypes = []
    lib.bdg_last_error.restype = C.c_char_p
    _lib = lib
    return lib


_pack = None


def pack_dict(entries: dict, keys: np.ndarray, vals: np.ndarray) -> int:
    """Write the ``((x,y,z),(x,y,z)) -> 2x2 complex128`` entries of a dict into ``keys [n,2,3] int64`` and
    ``vals [n,2,2] complex128`` with one C loop (``csrc/pack_dict.c``).  Returns the number of entries written,
    or a negative number if an entry is not of that plain form (the caller packs the dict with numpy instead);
    -1 also when the helper library has not been built (it is optional: a speed-up, not a code path of its own)."""
    global _pack
    if _pack is None:
        path = os.path.join(_PKG, "_bdgpack.so")
        if not os.path.exists(path):
            _pack = False
        else:
            lib = C.PyDLL(path)
            lib.bdg_pack_dict.argtypes = [C.py_object, _vp, _vp]
            lib.bdg_pack_dict.restype = C.c_longlong
            lib.bdg_pack_dict_cubic.argtypes = [C.py_object, C.c_longlong, C.c_longlong, C.c_longlong, _vp, _vp, _vp]
            lib.bdg_pack_dict_cubic.restype = C.c_longlong
            _pack = lib
    if _pack is False:
        return -1
    return int(_pack.bdg_pack_dict(entries, keys.ctypes.data_as(_vp), vals.ctypes.data_as(_vp)))


def pack_dict_cubic(entries: dict, shape, site_i: np.ndarray, site_j: np.ndarray, vals: np.ndarray) -> int:
    """``pack_dict`` for a stock ``CubicLattice(shape)``: the keys become flat int32 site indices in the same C loop."""
    if pack_dict({}, np.empty((0, 2, 3), np.int64), np.empty((0, 2, 2), np.complex128)) < 0:
        return -1
    return int(_pack.bdg_pack_dict_cubic(entries, int(shape[0]), int(shape[1]), int(shape[2]), site_i.ctypes.data_as(_vp),
                                         site_j.ctypes.data_as(_vp), vals.ctypes.data_as(_vp)))


def last_error() -> str:
    return load().bdg_last_error().decode("utf-8", "replace")


_EXC = {
    E_INVALID: ValueError,
    E_CUDA: RuntimeError,
    E_NOT_NEIGHBOUR: IndexError,
    E_NOT_HERMITIAN: RuntimeError,
    E_OUT_OF_BOUNDS: ValueError,
    E_NO_DEVICE: RuntimeError,
}


def check(rc: int):
    if rc != OK:
        raise _EXC.get(rc, RuntimeError)(last_error())


def release_cached(device: int = 0) -> None:
    """Return the library's cache of released device buffers to the CUDA driver."""
    check(load().bdg_release_cached(int(device)))


def cheb_moments_multi(systems, n_moments: int, *, probe_rows=None, n_random: int = 0, seed: int = 0, scale: float,
                       summed: bool = False) -> np.ndarray:
    """``bdg_cheb_moments_multi``: one process, one ``System`` (replica of the same Hamiltonian) per GPU; the columns
    are sharded over them and one NCCL collective combines the moments.  Returns ``[n_moments]`` (summed) or
    ``[n_moments, n_cols]``."""
    lib = load()
    handles = (_vp * len(systems))(*[s._h for s in systems])
    if probe_rows is not None:
        rows = _as(probe_rows, np.int64)
        kind, n_cols, rows_ptr = X0_PROBE, len(rows), _ptr(rows)
    else:
        kind, n_cols, rows_ptr = X0_RADEMACHER, int(n_random), None
    out = np.empty((n_moments,) if summed else (n_moments, n_cols), dtype=np.float64)
    check(lib.bdg_cheb_moments_multi(handles, len(systems), kind, n_cols, rows_ptr, C.c_uint64(int(seed)), float(scale),
                                     int(n_moments), MU_SUM if summed else MU_PER_COLUMN, _ptr(out)))
    return out


def device_count() -> int:
    n = C.c_int(0)
    rc = load().bdg_device_count(C.byref(n))
    return n.value if rc == OK else 0


def _ptr(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(_vp)


def _as_index(a, what="site index"):
    """int32 site indices for the ABI; wider integers are range-checked (no silent wrap), floats refused."""
    a = np.asarray(a)
    if a.dtype == np.int32:
        return np.ascontiguousarray(a)
    if a.size and a.dtype.kind not in "iu":
        raise TypeError(f"{what} arrays must be integers, got {a.dtype}")
    if a.size and (int(a.min()) < np.iinfo(np.int32).min or int(a.max()) > np.iinfo(np.int32).max):
        raise ValueError(f"{what} out of the int32 range of the BSR structure")
    return np.ascontiguousarray(a, dtype=np.int32)


def _as(a, dtype, shape_tail=()):
    a = np.ascontiguousarray(a, dtype=dtype)
    if shape_tail and a.shape[1:] != shape_tail:
        raise ValueError(f"expected trailing shape {shape_tail}, got {a.shape[1:]}")
    return a


class System:
    """Owner of one ``bdg_t`` handle (one Hamiltonian on one GPU)."""

    def __init__(self, handle, n_sites, n_blocks, device):
        self._h = handle
        self.n_sites = n_sites
        self.n_blocks = n_blocks
        self.device = device

    # -- construction / destruction ------------------------------------------------------
    @classmethod
    def _finish(cls, lib, handle, device):
        n, nb = C.c_int64(), C.c_int64()
        check(lib.bdg_skeleton_sizes(handle, C.byref(n), C.byref(nb)))
        return cls(handle, n.value, nb.value, device)

    @classmethod
    def cubic(cls, shape, device=0):
        lib = load()
        h = _vp()
        check(lib.bdg_create_cubic(device, int(shape[0]), int(shape[1]), int(shape[2]), C.byref(h)))
        return cls._finish(lib, h, device)

    @classmethod
    def generic(cls, n_sites, pair_i, pair_j, device=0):
        lib = load()
        pi, pj = _as_index(pair_i), _as_index(pair_j)
        h = _vp()
        check(lib.bdg_create_generic(device, int(n_sites), len(pi), _ptr(pi), _ptr(pj), C.byref(h)))
        return cls._finish(lib, h, device)

    def close(self):
        if self._h is not None and _lib is not None:
            _lib.bdg_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing ---------------------------------------------------------------------------
    def set_stream(self, stream_ptr: int | None):
        """Borrow a CUDA stream given as an integer handle (``torch.cuda.Stream.cuda_stream``);
        ``None`` restores the handle's own stream.  Handle 0 is CUDA's legacy default stream,
        which the C ABI spells ``cudaStreamLegacy`` (0x1) because NULL means "own stream"."""
        if stream_ptr is None:
            check(load().bdg_set_stream(self._h, None))
        else:
            check(load().bdg_set_stream(self._h, _vp(stream_ptr if stream_ptr != 0 else 1)))

    def sync(self):
        check(load().bdg_sync(self._h))

    def device_bytes(self) -> int:
        b = C.c_int64()
        check(load().bdg_device_bytes(self._h, C.byref(b)))
        return b.value

    # -- assembly -----------------------------------------------------------------------------
    def lookup(self, i, j) -> np.ndarray:
        i, j = _as_index(i), _as_index(j)
        k = np.empty(len(i), dtype=np.int64)
        bad = C.c_int64(-1)
        check(load().bdg_lookup(self._h, len(i), _ptr(i), _ptr(j), _ptr(k), C.byref(bad)))
        return k

    def scatter(self, h_i, h_j, h_val, p_i, p_j, p_val, herm_tol=1e-6) -> float:
        h_i, h_j = _as_index(h_i), _as_index(h_j)
        p_i, p_j = _as_index(p_i), _as_index(p_j)
        h_val = _as(np.asarray(h_val).reshape(-1, 2, 2), np.complex128, (2, 2))
        p_val = _as(np.asarray(p_val).reshape(-1, 2, 2), np.complex128, (2, 2))
        if not (len(h_i) == len(h_j) == len(h_val) and len(p_i) == len(p_j) == len(p_val)):
            raise ValueError("index and value arrays differ in length")
        dev, bad = C.c_double(0.0), C.c_int64(-1)
        check(load().bdg_scatter(self._h, len(h_i), _ptr(h_i), _ptr(h_j), _ptr(h_val), len(p_i), _ptr(p_i),
                                 _ptr(p_j), _ptr(p_val), float(herm_tol), C.byref(dev), C.byref(bad)))
        return dev.value

    def clear(self):
        check(load().bdg_clear(self._h))

    def stats(self) -> dict:
        """Counters of the rebuild / patch-in-place decisions (``bdg_stats``)."""
        out = (C.c_int64 * 5)()
        check(load().bdg_stats(self._h, out))
        return dict(zip(("compactions", "native_builds", "patched_scatters", "patched_blocks", "listed_hermitian_checks"), list(out)))

    def export_bsr(self, eliminate_zeros: bool):
        lib = load()
        nb = C.c_int64()
        check(lib.bdg_export_bsr(self._h, int(eliminate_zeros), C.byref(nb), None, None, None))
        indptr = np.empty(self.n_sites + 1, dtype=np.int32)
        indices = np.empty(nb.value, dtype=np.int32)
        data = np.empty((nb.value, 4, 4), dtype=np.complex128)
        check(lib.bdg_export_bsr(self._h, int(eliminate_zeros), C.byref(nb), _ptr(indptr), _ptr(indices), _ptr(data)))
        return indptr, indices, data

    def export_csr(self, transpose: bool = False):
        """(indptr, indices, data) of the CSR (or, transposed, CSC) form without explicit zeros."""
        lib = load()
        nnz = C.c_int64()
        indptr = np.empty(4 * self.n_sites + 1, dtype=np.int32)
        check(lib.bdg_export_csr(self._h, int(transpose), C.byref(nnz), _ptr(indptr), None, None))
        indices = np.empty(nnz.value, dtype=np.int32)
        data = np.empty(nnz.value, dtype=np.complex128)
        check(lib.bdg_export_csr(self._h, int(transpose), C.byref(nnz), _ptr(indptr), _ptr(indices), _ptr(data)))
        return indptr, indices, data

    def zero_scalar_rows(self) -> int:
        """Scalar rows of the 4N x 4N matrix without a single non-zero entry (the counting phase of ``bdg_export_csr``:
        only the 4N + 1 row offsets come back)."""
        nnz = C.c_int64()
        indptr = np.empty(4 * self.n_sites + 1, dtype=np.int32)
        check(load().bdg_export_csr(self._h, 0, C.byref(nnz), _ptr(indptr), None, None))
        return int(np.count_nonzero(np.diff(indptr) == 0))

    def export_dense(self) -> np.ndarray:
        out = np.empty((4 * self.n_sites, 4 * self.n_sites), dtype=np.complex128)
        check(load().bdg_export_dense(self._h, _ptr(out)))
        return out

    def import_data(self, data):
        data = _as(data, np.complex128)
        if data.shape != (self.n_blocks, 4, 4):
            raise ValueError(f"expected data of shape {(self.n_blocks, 4, 4)}, got {data.shape}")
        check(load().bdg_import_data(self._h, _ptr(data)))

    def norm_inf(self) -> float:
        v = C.c_double()
        check(load().bdg_norm_inf(self._h, C.byref(v)))
        return v.value

    # -- Chebyshev engine ---------------------------------------------------------------------
    def cheb_begin(self, *, probe_rows=None, n_random=0, seed=0, col_offset=0, scale, kernel="auto"):
        lib = load()
        if probe_rows is not None:
            rows = _as(probe_rows, np.int64)
            check(lib.bdg_cheb_begin(self._h, X0_PROBE, len(rows), _ptr(rows), 0, 0, float(scale), KERNELS[kernel]))
        else:
            check(lib.bdg_cheb_begin(self._h, X0_RADEMACHER, int(n_random), None, C.c_uint64(int(seed)),
                                     int(col_offset), float(scale), KERNELS[kernel]))

    def cheb_steps(self, n_steps: int, timed: bool = False):
        ms = C.c_float(0.0)
        check(load().bdg_cheb_steps(self._h, int(n_steps), C.byref(ms) if timed else None))
        return ms.value if timed else None

    def cheb_reserve(self, n_steps: int):
        check(load().bdg_cheb_reserve(self._h, int(n_steps)))

    def cheb_available(self) -> int:
        n = C.c_int32()
        check(load().bdg_cheb_available(self._h, C.byref(n)))
        return n.value

    def cheb_read(self, n_moments: int, n_cols: int, summed: bool = False, device_ptr: int | None = None):
        """Moments as ``[n_moments, n_cols]`` (or ``[n_moments]`` summed over columns); with
        ``device_ptr`` they are written to that device address instead and ``None`` is returned."""
        lib = load()
        if device_ptr is not None:
            check(lib.bdg_cheb_moments_read(self._h, int(n_moments), int(summed), _vp(device_ptr), 1))
            return None
        out = np.empty((n_moments,) if summed else (n_moments, n_cols), dtype=np.float64)
        check(lib.bdg_cheb_moments_read(self._h, int(n_moments), int(summed), _ptr(out), 0))
        return out

    def cheb_vectors(self, n_cols: int, which: int = 0) -> np.ndarray:
        out = np.empty((4 * self.n_sites, n_cols), dtype=np.complex128)
        check(load().bdg_cheb_vectors(self._h, int(which), _ptr(out)))
        return out

    def cheb_format(self) -> dict:
        """Kernel / matrix format the active recursion runs on (``kernel="auto"`` resolved)."""
        k, mb, nu = C.c_int32(), C.c_int64(), C.c_int64()
        check(load().bdg_cheb_format(self._h, C.byref(k), C.byref(mb), C.byref(nu)))
        return {"kernel": KERNEL_NAMES[k.value], "matrix_bytes_per_step": mb.value, "distinct_blocks": nu.value}

    def cheb_launched(self) -> list[str]:
        """Names of the recursion kernels the current recursion has launched (``bdg_cheb_launched``), as
        ``cudaFuncGetName`` gives them, in the order of their first launch."""
        lib = load()
        needed = C.c_int64()
        check(lib.bdg_cheb_launched(self._h, None, 0, C.byref(needed)))
        buf = C.create_string_buffer(needed.value)
        check(lib.bdg_cheb_launched(self._h, buf, needed.value, C.byref(needed)))
        text = buf.value.decode("utf-8")
        return text.split("\n") if text else []

    def cheb_info(self) -> dict:
        nb, by, la = C.c_int64(), C.c_int64(), C.c_int64()
        pw, npan = C.c_int32(), C.c_int32()
        check(load().bdg_cheb_info(self._h, C.byref(nb), C.byref(by), C.byref(pw), C.byref(npan), C.byref(la)))
        return dict(n_blocks=nb.value, bytes_per_step=by.value, panel_width=pw.value, n_panels=npan.value,
                    launches=la.value)

    def cheb_end(self):
        check(load().bdg_cheb_end(self._h))

    # -- observables evaluated on the device from the current recursion's moments -----------------
    def kpm_resolvent(self, n_moments: int, n_cols: int, w, pref) -> np.ndarray:
        """``g[c, e] = pref[e] * sum_n (2 - δ_n0) mu_n[c] w[e]**n`` as complex ``[n_cols, len(w)]``."""
        w, pref = _as(w, np.complex128), _as(pref, np.complex128)
        if w.shape != pref.shape or w.ndim != 1:
            raise ValueError("w and pref must be 1-D arrays of equal length")
        out = np.empty((n_cols, len(w)), dtype=np.complex128)
        check(load().bdg_kpm_resolvent(self._h, int(n_moments), len(w), _ptr(w), _ptr(pref), _ptr(out), 0))
        return out

    def kpm_contract(self, coef, n_cols: int, summed: bool = False):
        """``sum_n coef[n] mu_n[c]`` per column (``[n_cols]``) or summed over the columns (float)."""
        coef = _as(coef, np.float64)
        out = np.empty(1 if summed else n_cols, dtype=np.float64)
        check(load().bdg_kpm_contract(self._h, len(coef), _ptr(coef), int(summed), _ptr(out), 0))
        return float(out[0]) if summed else out

    def cheb_local_begin(self, coef, cols, sites):
        """Register the local accumulator on the active recursion (``bdg_cheb_local_begin``): series ``coef``, reads
        ``(cols[r], sites[r])``.  Adds the ``T_0`` and ``T_1`` terms; the rest arrive with ``cheb_steps``."""
        coef = _as(coef, np.float64)
        cols, sites = _as_index(cols, "column index"), _as_index(sites)
        if coef.ndim != 1 or cols.shape != sites.shape or cols.ndim != 1:
            raise ValueError("coef, cols and sites must be 1-D, cols and sites of equal length")
        check(load().bdg_cheb_local_begin(self._h, len(coef), _ptr(coef), len(cols), _ptr(cols), _ptr(sites)))

    def cheb_local_read(self, n_reads: int, device_ptr: int | None = None):
        """The accumulated ``[n_reads, 4]`` complex values; with ``device_ptr`` they are written to that device address
        instead (``n_reads * 64`` bytes) and ``None`` is returned."""
        if device_ptr is not None:
            check(load().bdg_cheb_local_read(self._h, _vp(device_ptr), 1))
            return None
        out = np.empty((n_reads, 4), dtype=np.complex128)
        check(load().bdg_cheb_local_read(self._h, _ptr(out), 0))
        return out
