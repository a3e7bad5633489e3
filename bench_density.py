"""Benchmark of the local density matrix / s-wave order parameter (``Hamiltonian.order_parameter``) on one GPU.

Prints one JSON line: the device and its power limit; at C2 (README model, 100 x 100 sites, one probe column per
site = 10^4 columns) the recursion time with and without the local accumulator on the same columns (alternated,
windows of >= 1 s); the time per ``order_parameter`` call at C1 (40 x 40, 1600 columns) and C2; the dense
alternative at C1, ``torch.linalg.eigh`` of the 6400 x 6400 matrix on the same GPU; and the largest difference
between the KPM and the dense order parameter at C1.

``--spacing S [S ...]`` measures instead ``order_parameter`` over every site of the README model on 1000 x 1000 sites
from distance-classed columns (``spacing=S``, one column per class): seconds per call for each spacing, and the largest
deviation from the one-column-per-site path at 50 sampled sites.

    python bench_density.py [--temperature 0.1] [--repeats 3] [--device 0] [--spacing 8 16]

It writes nothing into the tree.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def device_info(dev: int) -> dict:
    import torch

    info = {"device": torch.cuda.get_device_name(dev)}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={dev}", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        power, clock = (v.strip() for v in out.strip().splitlines()[0].split(","))
        info.update(power_limit_w=float(power), clocks_max_sm_mhz=float(clock))
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        info.update(power_limit_w=None, clocks_max_sm_mhz=None)
    return info


def readme_system(L: int, dev: int):
    import bodge_b200 as b
    from bodge_b200 import workloads

    system = b.Hamiltonian(b.CubicLattice((L, L, 1)), device=dev)
    system.fill(*workloads.readme_swave((L, L, 1)))
    return system


def recursion_seconds(system, rows, scale, steps, coef=None) -> float:
    """Device time of ``steps`` recursion steps on the probe columns ``rows``, with the local accumulator (one read per
    column, at the column's own site) when ``coef`` is given."""
    sysn = system._sys
    sysn.cheb_begin(probe_rows=rows, scale=scale, kernel="auto")
    if coef is not None:
        sysn.cheb_local_begin(coef, np.arange(len(rows)), rows // 4)
    return sysn.cheb_steps(steps, timed=True) / 1e3


def timed_call(fn, repeats: int) -> list[float]:
    fn()  # warm-up: module loads, buffer allocation
    out = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        out.append(time.perf_counter() - t0)
    return out


def spacing_case(dev: int, T: float, spacings, repeats: int) -> dict:
    """``order_parameter`` over every site of the 1000 x 1000 README model with ``spacing=s``: seconds per call (every
    call, the first included) and the largest deviation from the exact path at 50 sampled sites."""
    from bodge_b200 import kpm

    system = readme_system(1000, dev)
    n = system.lattice.size
    scale = system.spectral_bound()
    sample = np.sort(np.random.default_rng(7).choice(n, 50, replace=False))
    coords = [tuple(int(v) for v in c) for c in system.lattice.sites_array()[sample]]
    t0 = time.perf_counter()
    exact = system.order_parameter(T, 1.0, sites=coords)
    out = {"sites": n, "n_coef": kpm.free_energy_moments(T, scale)[0], "scale": scale, "sampled_sites": len(sample),
           "exact_sampled_s": time.perf_counter() - t0, "spacing": {}}
    for s in spacings:
        per_call = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            delta = system.order_parameter(T, 1.0, spacing=s)
            per_call.append(time.perf_counter() - t0)
        out["spacing"][str(s)] = {"classes": int(system._classes(s).max()) + 1, "per_call_s": per_call,
                                  "max_abs_dev_sampled": float(np.max(np.abs(delta[sample] - exact))),
                                  "delta_range": [float(np.min(np.abs(delta))), float(np.max(np.abs(delta)))]}
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--temperature", type=float, default=0.1)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--spacing", type=int, nargs="+", default=None,
                    help="measure order_parameter(spacing=S) on 1000 x 1000 sites for each S instead")
    args = ap.parse_args()

    import torch

    from bodge_b200 import _native, kpm

    if not torch.cuda.is_available() or _native.device_count() == 0:
        raise SystemExit("bench_density.py needs a CUDA device")
    dev, T, reps = args.device, args.temperature, args.repeats
    result = device_info(dev)
    result.update(model="readme_swave", temperature=T, potential=1.0)
    if args.spacing:
        result["order_parameter_spacing"] = spacing_case(dev, T, args.spacing, reps)
        print(json.dumps(result))
        return

    # --- C2: accumulator overhead on the recursion, then order_parameter end to end ---------------------------------
    c2 = readme_system(100, dev)
    scale = c2.spectral_bound()
    n_coef = kpm.free_energy_moments(T, scale)[0]
    rows = 4 * np.arange(c2.lattice.size, dtype=np.int64) + 3
    pilot = recursion_seconds(c2, rows, scale, 64)
    steps = max(n_coef - 1, int(np.ceil(1.05 * 64 / pilot)))  # a window of >= 1 s
    steps += steps & 1
    coef = kpm.fermi_coefficients(T, steps + 1, scale)  # every timed step adds its term
    plain, accum = [], []
    for _ in range(reps):
        plain.append(recursion_seconds(c2, rows, scale, steps))
        accum.append(recursion_seconds(c2, rows, scale, steps, coef))
    kernel = c2._sys.cheb_format()["kernel"]
    result["c2_recursion"] = {
        "sites": c2.lattice.size, "columns": len(rows), "kernel": kernel, "steps": steps,
        "plain_s": plain, "accumulator_s": accum,
        "overhead": float(np.median(accum) / np.median(plain) - 1.0),
    }
    op_c2 = timed_call(lambda: c2.order_parameter(T, 1.0), reps)
    result["order_parameter_s"] = {"C2": {"sites": c2.lattice.size, "n_coef": n_coef, "scale": scale, "per_call": op_c2}}
    del c2
    _native.release_cached(dev)

    # --- C1: order_parameter, the dense alternative, and their agreement ---------------------------------------------
    c1 = readme_system(40, dev)
    scale1 = c1.spectral_bound()
    op_c1 = timed_call(lambda: c1.order_parameter(T, 1.0), reps)
    delta_kpm = c1.order_parameter(T, 1.0)
    result["order_parameter_s"]["C1"] = {"sites": c1.lattice.size, "n_coef": kpm.free_energy_moments(T, scale1)[0],
                                         "scale": scale1, "per_call": op_c1}
    H = torch.as_tensor(np.asarray(c1.matrix("dense")), device=torch.device("cuda", dev))
    eig = {}

    def dense():
        eig["w"], eig["v"] = torch.linalg.eigh(H)
        torch.cuda.synchronize(dev)

    result["eigh_c1_s"] = timed_call(dense, reps)
    w, v = eig["w"], eig["v"]
    f = torch.special.expit(-w / T)
    rho_03 = ((v[0::4] * f) * v[3::4].conj()).sum(dim=1)  # rho[4i, 4i+3] = sum_k U[4i,k] f_k conj(U[4i+3,k])
    delta_dense = (-1.0 * rho_03).cpu().numpy()
    result["parity_c1_max_abs"] = float(np.max(np.abs(delta_kpm - delta_dense)))
    result["delta_c1_range"] = [float(np.min(np.abs(delta_kpm))), float(np.max(np.abs(delta_kpm)))]
    print(json.dumps(result))


if __name__ == "__main__":
    main()
