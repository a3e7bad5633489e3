"""Distance classes of the sites of a ``CubicLattice`` for probing many sites with few Chebyshev columns.

A polynomial ``p`` of degree ``m`` has ``p(H̃)[4i+α, 4j+β] = 0`` whenever sites ``i`` and ``j`` are more than ``m`` hops
apart in the graph of the stored blocks.  If the sites are split into classes whose distinct members are at least
``spacing`` hops apart, one start column per (class ``k``, component ``β``), ``x = Σ_{j in class k} e_{4j+β}``, read at
a site ``i`` of that class gives ``p(H̃)[4i+α, 4i+β]`` plus the elements between ``i`` and the other sites of its class:
exactly zero when ``spacing > m``, and otherwise elements of ``f(H)`` at least ``spacing`` hops away, which decay
exponentially with distance for the Fermi function at T > 0.  ``Hamiltonian.density_matrix(spacing=...)`` and friends
use these classes (``bdg_set_classes`` / ``BDG_X0_CLASS`` in ``include/bdg.h``).

The classes are built per axis, and a site's class is the tuple of its three axis classes.  Each axis rule gives two
distinct coordinates of one class a (cyclic, if the axis wraps) distance of at least ``spacing``, so two distinct sites
of one class are at least that many hops apart:

* open axis: ``x mod s``; with ``L <= s`` every coordinate is its own class;
* wrapping axis with ``L >= s``: ``g = L // s`` consecutive runs of ``L // g`` or ``L // g + 1`` coordinates, the class
  being the offset inside the run (``x mod s`` is wrong when ``s`` does not divide ``L``: the last and the first run
  would be too close across the wrap); ``ceil(L / g)`` classes;
* wrapping axis with ``L < s``: one class per coordinate.
"""

from __future__ import annotations

import numpy as np


def axis_classes(length: int, spacing: int, wraps: bool) -> np.ndarray:
    """Class of every coordinate ``0 .. length - 1`` of one axis (int64), by the rule in the module docstring."""
    L, s = int(length), int(spacing)
    if L < 1 or s < 1:
        raise ValueError(f"need a positive axis length and spacing, got {L} and {s}")
    x = np.arange(L, dtype=np.int64)
    if not wraps:
        return x % s
    if L < s:
        return x
    g = L // s
    base, extra = divmod(L, g)  # the first `extra` runs are one longer
    lengths = np.array([base + 1] * extra + [base] * (g - extra), dtype=np.int64)
    starts = np.cumsum(lengths) - lengths
    return x - np.repeat(starts, lengths)


def site_classes(shape, spacing: int, wraps) -> tuple[np.ndarray, int]:
    """``(class of every site in flat-index order as int32, number of classes)`` for ``CubicLattice(shape)``, whose flat
    index is ``z + Lz*(y + Ly*x)``; ``wraps[a]``: whether axis ``a`` has a non-zero block between its two faces."""
    per_axis = [axis_classes(L, spacing, w) for L, w in zip(shape, wraps)]
    counts = [int(c.max()) + 1 for c in per_axis]
    cx, cy, cz = per_axis
    cls = (cx[:, None, None] * counts[1] + cy[None, :, None]) * counts[2] + cz[None, None, :]
    n_classes = counts[0] * counts[1] * counts[2]
    if n_classes >= 2**31:
        raise ValueError(f"{n_classes} classes do not fit the int32 class index")
    return cls.astype(np.int32).ravel(), n_classes
