"""Scripted sequences of small scatters that ``bdg_scatter`` patches into the step kernels' copies of the matrix in place
(``csrc/formats.cu``: ``ell_patch`` / ``patch_blocks``), or that must take the rebuild path.

Each geometry x model pair gets one sequence, applied in order to one system built by ``variant_cases.build``.  A step
is one packed ``fill`` tuple with the path it must take ("patch" or "rebuild"), whether the stored matrix is Hermitian
after it, and, where it is pinned, how many entries it adds to the block dictionary.  The labels are derived from the
matrix as the sequence goes (``_label``), not from the model name.  The oracle state after every step is kept with it:
``test_patch_cases.py`` checks the sequences on the CPU, ``test_gpu_patch.py`` runs them on the GPU.

What each geometry's patch must keep current besides the compacted ``packed`` data:

* ``chain``      fixed-width rows and dictionary only (M < 3: no plane codes);
* ``square``     plane codes of the two-steps-per-pass kernel, open stencil;
* ``pair_torus`` plane codes with in-plane and x wrap-around;
* ``slab``       cube codes with Lz = 2 (``diag`` / ``normal``: the cube kernel needs real-diagonal hopping);
* ``cube3d``     cube codes (``t2`` on 4-column panels);
* ``hub8``       a generic lattice: dictionary at width 8, no direction codes;
* ``hub41``      rows of 41 blocks: no fixed-width copy, only ``packed`` is patched (DMMA, FMA).
"""

from __future__ import annotations

import zlib
from dataclasses import dataclass

import numpy as np

import cases
import variant_cases as vc
from oracle import bdg_oracle as orc

MODELS = ("diag", "normal", "gen", "pairgen")
SEQUENCES = [(g, m) for g in ("chain", "square", "pair_torus", "hub8", "hub41") for m in MODELS] + \
            [(g, m) for g in ("slab", "cube3d") for m in ("diag", "normal")]
NO_DICTIONARY = ("hub41",)   # rows wider than 8 blocks: no fixed-width copy, so no dictionary and no kernel flags


@dataclass
class Step:
    name: str
    packed: tuple               # (h_i, h_j, h_val, p_i, p_j, p_val) as ``Hamiltonian.fill`` takes them
    path: str                   # "patch" or "rebuild"
    hermitian: bool             # the stored matrix after the step
    new_entries: int | None     # growth of the dictionary's distinct blocks when pinned (dictionary geometries only)
    data: np.ndarray            # oracle skeleton data after the step

    @property
    def n_written(self):
        """Skeleton blocks the scatter writes: one per H entry, two per Δ entry (``patched_blocks``)."""
        return len(self.packed[0]) + 2 * len(self.packed[3])


@dataclass
class Sequence:
    geometry: str
    model: str
    indptr: np.ndarray
    indices: np.ndarray
    initial: np.ndarray         # oracle skeleton data of the built system
    steps: list

    @property
    def dictionary(self):
        return self.geometry not in NO_DICTIONARY


# ---- block properties over the oracle skeleton ------------------------------------------------------------------------
def block_rows(indptr):
    return np.repeat(np.arange(len(indptr) - 1), np.diff(indptr))


def real_diagonal(blocks):
    """Per 4x4 block: real and diagonal (every off-diagonal entry and every imaginary part == 0)."""
    blocks = np.asarray(blocks)
    off = blocks * (1 - np.eye(4))
    return ~((off != 0).any(axis=(1, 2)) | (blocks.imag != 0).any(axis=(1, 2)))


def nonzero(data):
    return (np.asarray(data) != 0).reshape(len(data), -1).any(axis=1)


def offsite_real_diagonal(indptr, indices, data):
    """Every non-zero off-site block is real-diagonal."""
    off = (block_rows(indptr) != indices) & nonzero(data)
    return bool(real_diagonal(data[off]).all())


def onsite_real_diagonal(indptr, indices, data):
    on = (block_rows(indptr) == indices) & nonzero(data)
    return bool(real_diagonal(data[on]).all())


def hermitian(indptr, indices, data):
    return orc.hermitian_deviation(indptr, indices, data) == 0.0


# ---- packed tuples ---------------------------------------------------------------------------------------------------
def _i(v):
    return np.asarray(v, dtype=np.int32).reshape(-1)


def _m(v):
    return np.asarray(v, dtype=np.complex128).reshape(-1, 2, 2)


def packed(h=(), p=()):
    """``h`` / ``p``: lists of ``(i, j, 2x2)`` H and Δ entries (flat site indices)."""
    h, p = list(h), list(p)
    return (_i([e[0] for e in h]), _i([e[1] for e in h]), _m([e[2] for e in h]),
            _i([e[0] for e in p]), _i([e[1] for e in p]), _m([e[2] for e in p]))


def _label(seq_dict, diag_flag, before, after, indptr, indices):
    """The path ``bdg_scatter`` must take: rebuild when the zero pattern changes, or when an off-site block that is not
    real-diagonal is written while the dictionary's DIAG flag holds; the flag is re-derived at each rebuild."""
    if not np.array_equal(nonzero(before), nonzero(after)):
        return "rebuild"
    if seq_dict and diag_flag and not offsite_real_diagonal(indptr, indices, after):
        return "rebuild"
    return "patch"


# ---- the sequences ---------------------------------------------------------------------------------------------------
def _skeleton(lattice):
    from bodge_b200.lattice import CubicLattice

    if type(lattice) is CubicLattice:
        return orc.cubic_skeleton(lattice.shape)
    pairs = [(lattice[ri], lattice[rj]) for ri, rj in lattice]
    return orc.skeleton_from_pairs(lattice.size, [a for a, _ in pairs], [b for _, b in pairs])


def sequence(geometry, model) -> Sequence:
    api = cases.recorder_api()
    σ0, σ1, σ3, jσ2 = api.σ0, api.σ1, api.σ3, api.jσ2
    lattice, pairs = vc.lattice_pairs(api, geometry)
    recorder = vc.fill(api, api.Hamiltonian(lattice), pairs, model)
    indptr, indices = _skeleton(lattice)
    data = orc.scatter(indptr, indices, orc.zero_data(indices), *recorder.packed())
    initial = data.copy()
    n = lattice.size
    n_blocks = len(indices)
    rng = np.random.default_rng(zlib.crc32(f"{geometry}-{model}".encode()))
    nbrs = {i: set() for i in range(n)}
    for a, b in pairs:
        if a != b:
            nbrs[lattice[a]].add(lattice[b])
            nbrs[lattice[b]].add(lattice[a])
    bonds = sorted({(min(a, b), max(a, b)) for a in nbrs for b in nbrs[a]})
    order = rng.permutation(n)
    u1, u2, u3 = (sorted(int(s) for s in order[3 * k:3 * k + 3]) for k in range(3))
    center = n // 2 if geometry.startswith("hub") else lattice.index(tuple(s // 2 for s in lattice.shape))
    onsite0 = 3.0 * σ0 - 0.05 * σ3   # vc.fill's on-site H

    writes = []   # (name, packed, new_entries)
    # U1: new real-diagonal on-site values, all distinct
    writes.append(("U1", packed(h=[(s, s, (2.0 + 0.1 * k) * σ0 - 0.3 * σ3) for k, s in enumerate(u1)]), None))
    # U2: an in-plane field on a few sites: the on-site blocks are no longer real-diagonal (the SD kernels must drop out)
    writes.append(("U2", packed(h=[(s, s, onsite0 + 0.4 * σ1) for s in u2]), None))
    # U3: on-site pairing on a few sites (the pairing list: two klists per scatter, here the same block twice)
    writes.append(("U3", packed(p=[(s, s, -(0.15 + 0.05 * k) * jσ2) for k, s in enumerate(u3)]), None))
    # U4: a new real-diagonal bond value in every stencil direction of two sites, both orientations (site 0 of a torus
    # reaches its neighbours across both wrap-around edges); rows of more than a few blocks are cut to the quarter rule
    u4 = [(0, j) for j in sorted(nbrs[0])] + [(center, j) for j in sorted(nbrs[center]) if j != 0]
    u4 = u4[:max(1, n_blocks // 10)]
    writes.append(("U4", packed(h=[e for i, j in u4 for e in ((i, j, -1.3 * σ0), (j, i, -1.3 * σ0))]), None))
    used = {frozenset(b) for b in u4}
    free = [b for b in bonds if frozenset(b) not in used]
    b5, b6, b10 = free[len(free) // 3], free[len(free) // 2], free[(2 * len(free)) // 3]
    # U5: a complex bond value and its conjugate transpose
    hop = -1.0 * σ0 + 0.2j * σ1
    writes.append(("U5", packed(h=[(b5[0], b5[1], hop), (b5[1], b5[0], hop.conj().T)]), None))
    # U6: bond pairing in both directions
    writes.append(("U6", packed(p=[(b6[0], b6[1], -0.1 * jσ2), (b6[1], b6[0], -0.1 * jσ2)]), None))
    # U7: the same values again: no new dictionary entry
    writes.append(("U7", writes[-1][1], 0))
    # U8: a block back to its build-time value: the lookup finds the original entry
    writes.append(("U8", packed(h=[(u1[0], u1[0], onsite0)]), 0))
    # U9: an eighth of all sites get one common new on-site block in one scatter (concurrent insert-and-wait); the
    # pairing-patched sites of U3 are left out, so that every written block is the same
    u9 = [int(s) for s in order[9:] if int(s) not in u3][:max(1, n // 8)]
    writes.append(("U9", packed(h=[(s, s, 2.7 * σ0 + 0.15 * σ3) for s in u9]), 1))
    # U10: a one-sided bond write (not Hermitian: the listed check raises, the matrix and the copies stay modified),
    # then the Hermitian rewrite, checked in full
    writes.append(("U10", packed(h=[(b10[0], b10[1], -0.7 * σ0)]), None))
    writes.append(("U10h", packed(h=[(b10[0], b10[1], -0.7 * σ0), (b10[1], b10[0], -0.7 * σ0)]), None))
    # U11: a block set to zero changes the zero pattern
    writes.append(("U11", packed(h=[(u1[1], u1[1], 0.0 * σ0)], p=[(u1[1], u1[1], 0.0 * jσ2)]), None))

    seq_dict = geometry not in NO_DICTIONARY
    diag_flag = offsite_real_diagonal(indptr, indices, data)
    steps = []
    for name, pk, new_entries in writes:
        after = orc.scatter(indptr, indices, data.copy(), *pk)
        path = _label(seq_dict, diag_flag, data, after, indptr, indices)
        if path == "rebuild":
            diag_flag = offsite_real_diagonal(indptr, indices, after)
        steps.append(Step(name, pk, path, hermitian(indptr, indices, after), new_entries, after))
        data = after
    return Sequence(geometry, model, indptr, indices, initial, steps)
