#!/usr/bin/env python
"""Benchmark of the hot path: fused Chebyshev H·X steps on a 10^6-site BdG Hamiltonian.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C5] [--cols 8]

One "step" = one application of H~ in the recursion T_{n+1} = 2 H~ T_n - T_{n-1} (+ the two moment dot
products) over one tile of ``cols`` vectors (default 8) per GPU.  The default kernel on the headline workload
(``t2``) does TWO steps per launch (``roofline.steps_per_launch``).  Workload: BASELINE.json config C5,
CubicLattice((1000,1000,1)) altermagnet/superconductor Josephson junction, 10^6 sites, 4,996,000 BSR blocks,
synthetic (SURVEY 8d).  N > 1: one process per GPU (torchrun), a replica of the matrix and its own 8 columns on
every GPU (weak scaling), one NCCL all-reduce of the moments at the end of the timed region.

Timed region: W warm-up steps, then K steps between two CUDA events on the launch stream; barrier + synchronize on
both sides, max over ranks.  ``steps`` echoes K, ``timed_steps`` counts the steps the region ran (K, or K + 1 for an
odd K on a kernel that advances two steps per launch).  The comparison runs and extras time K steps each as well.

``--dump-outputs DIR``: after the timed steps, the moments the headline recursion has computed are written as
``DIR/*.npy`` (float64, see ``dump_moments``); the inputs are fixed by the arguments, so two builds run with the same
arguments can be compared output for output.

Prints ONE JSON line.  ``value`` = whole-job steps/s with everything resident in HBM; ``e2e`` = the same metric
through the public API with the Hamiltonian terms in pinned HOST memory (upload + scatter + recursion + moments
back to the host inside the timed region); ``roofline`` = the dominant kernel against the measured HBM peak,
``frac`` on the bytes it MOVES (ncu DRAM bytes of the committed capture when there is one, else the format's own
accounting), the SURVEY-8d algorithmic-bytes figure beside it as ``speedup_vs_one_pass_roofline``;
``block_repetition`` = the same lattice with 10^6 distinct on-site blocks and with every block distinct;
``other_configs`` = BASELINE configs C2, C3, C4; ``strong_scaling`` = 64 columns in total; ``incremental_update`` = cost of
the reference's parameter-sweep idiom (re-enter ``with``, start the next recursion), patched vs rebuilt; ``parity_check`` =
the first moments against the CPU oracle (N = 1) / against a single-GPU recomputation of all shards (N > 1);
``cpu_baseline`` = scipy's bsr_matvecs recursion on the host cores (oracle port).

``--impl reference`` times only that CPU path (rank 0), on the same config/metric/unit.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the bench leaves the tree as it found it (it may be read-only)

import numpy as np  # noqa: E402

METRIC = "chebyshev_spmm_steps_per_s"
UNIT = "steps/s"
FALLBACK_HBM_GBS = 6650.0
DUMP_BYTES = 64 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000, help="timed steps of every recursion timing")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C5")
    ap.add_argument("--cols", type=int, default=8, help="vector columns per GPU (weak scaling, the default)")
    ap.add_argument("--total-cols", type=int, default=0,
                    help="strong scaling instead: this many columns in total, split evenly over the GPUs (SURVEY 8e: 64)")
    ap.add_argument("--kernel", default="auto_moments",
                    help="auto_moments = what chebyshev_moments / free_energy / ldos use (only moments are read)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-plain", action="store_true", help="skip the uncompressed-matrix / three-term comparison runs")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip block_repetition, other_configs and strong_scaling (only run with the default C5 headline)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the moments of the timed recursion to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    return args


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def recorded_traffic(workload_key):
    """DRAM bytes per launch of the step kernel from the committed ncu capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh).get(workload_key)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi sampled in the background during the timed region."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, watts, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            try:
                watts.append(float(r[2]))
            except (ValueError, IndexError):
                pass
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "sm_mhz_min": min(sm), "power_w": statistics.median(watts) if watts else None}


def workload_config(cfg_key, cfg, n_sites, n_blocks, cols):
    """The `config` object: the WORKLOAD only, identical for both arms (what ran it goes under `run`)."""
    vec_gb = 2 * 64 * n_sites * cols / 1e9
    return {"workload": cfg["label"], "config": cfg_key, "n_sites": n_sites, "n_blocks": n_blocks, "cols_per_gpu": cols,
            "l2": f"BSR matrix {260 * n_blocks / 1e9:.2f} GB + two vector sets {vec_gb:.2f} GB per GPU against a 126 MB L2"
                  + ("; inputs exceed L2, no flush needed" if 260 * n_blocks + vec_gb * 1e9 > 4 * 126e6 else "; L2-resident working set (SURVEY H5)")}


# ------------------------------------------------------------------------------------------
# reference arm / CPU baseline: scipy bsr_matvecs recursion on the host (oracle port)
# ------------------------------------------------------------------------------------------
def cpu_chebyshev(cfg_key, cols, steps, warmup, budget_s, moments_for_parity=0):
    from bodge_b200 import workloads
    from oracle import bdg_oracle as orc
    from oracle import cpu_baseline as cb

    cfg = workloads.CONFIGS[cfg_key]
    t0 = time.perf_counter()
    packed = cfg["build"](cfg["shape"])
    ptr, idx, dat = cb.assemble(cfg["shape"], packed)
    t_asm = time.perf_counter() - t0
    scale = 1.01 * orc.norm_inf(ptr, idx, dat)
    x0 = orc.rademacher(1234, 4 * (len(ptr) - 1), np.arange(cols))
    res = cb.time_steps(ptr, idx, dat, scale, x0, steps=steps, warmup=warmup, budget_s=budget_s)
    res["assembly_s"] = t_asm
    res["n_sites"] = len(ptr) - 1
    res["n_blocks"] = len(idx)
    res["scale"] = scale
    if moments_for_parity:
        # the checker: the first moments of the same columns by the oracle's three-term recursion, all host cores
        t0 = time.perf_counter()
        res["moments"] = cb.moments_parallel(ptr, idx, dat, scale, x0, moments_for_parity)
        res["moments_s"] = time.perf_counter() - t0
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from bodge_b200 import workloads

    cfg = workloads.CONFIGS[args.config]
    res = cpu_chebyshev(args.config, args.cols, args.steps, args.warmup, budget_s=120.0)
    value = 1e3 / res["ms_per_step"]
    sample = (f"{args.steps} steps after {args.warmup} warm-up on {res['fraction']:.3f} of the block rows per step "
              f"(time scaled to a full step), k={args.cols}, rows split over {res['cores']} processes")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.config, cfg, res["n_sites"], res["n_blocks"], args.cols),
        "run": {"what": "scipy bsr_matvecs recursion 2*(H~@T1)-T0 on the host (oracle port of the reference path; the reference "
                        "has no Chebyshev entry point, SURVEY 0.2)",
                "note": "the value is per 8-column tile; at N > 1 the GPU arm advances N such tiles at once, the host would run them "
                        "one after the other at this same rate"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": res["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
KERNEL_NAMES = {
    "t2": "cheb_pair_step<MODE=T2> (two applications of H~ per launch on the even vectors E_j = T_2j x: "
          "E_{j+1} = 2 T_2(H~) E_j - E_{j-1}; block-dictionary matrix, E_j planes staged in shared memory by TMA "
          "bulk copies, H~ E_j kept in shared memory, E_{j+1} written over E_{j-1})",
    "pair": "cheb_pair_step (two steps per launch: block-dictionary matrix, T_n planes staged in shared memory by "
            "TMA bulk copies, T_{n-1} straight to registers, T_{n+1} kept in shared memory)",
    "dict": "cheb_step_ell<DICT> (block-dictionary matrix)",
    "dict_diag": "cheb_step_ell<DICT,DIAG> (block-dictionary matrix, real-diagonal hopping blocks by DFMA)",
    "ell": "cheb_step_ell (every block from HBM)", "dmma": "cheb_step_dmma", "fma": "cheb_step_fma",
}
VECTOR_PASSES = {"pair": 128, "t2": 96}  # bytes per site, column and STEP (single-step kernels: 192)


def dict_api_assembly(b, device):
    """BASELINE config C2 through the reference's own surface -- ``with system as (H, Δ)`` and two
    Python loops (README.md:73-86) -- to ``matrix("bsr")``.  The user's loops are interpreter time
    no library can remove (SURVEY H1); ``library_s`` is everything else (skeleton, dict packing,
    H2D, scatter + symmetry fill + Hermitian check, zero-block compaction, D2H of the BSR arrays)."""
    warm = b.Hamiltonian(b.CubicLattice((4, 4, 1)), device=device)   # untimed: lazy loading of the packer, first allocations
    with warm as (H, D):
        H[(0, 0, 0), (0, 0, 0)] = 1.0 * b.σ0
    warm.matrix("bsr")
    del warm
    shape = (100, 100, 1)
    t0 = time.perf_counter()
    lattice = b.CubicLattice(shape)
    system = b.Hamiltonian(lattice, device=device)
    t1 = time.perf_counter()
    with system as (H, D):
        for i in lattice.sites():
            H[i, i] = 3.0 * b.σ0 - 0.05 * b.σ3
            D[i, i] = -0.10 * b.jσ2
        for i, j in lattice.bonds():
            H[i, j] = -1.0 * b.σ0
        t2 = time.perf_counter()
    t3 = time.perf_counter()
    bsr = system.matrix("bsr")
    t4 = time.perf_counter()
    return {"config": "C2 CubicLattice((100,100,1)) README s-wave via the dict API", "n_sites": lattice.size,
            "n_blocks": int(len(bsr.indices)), "sites_per_s": lattice.size / (t4 - t0),
            "library_sites_per_s": lattice.size / ((t1 - t0) + (t3 - t2) + (t4 - t3)),
            "user_loop_s": t2 - t1, "skeleton_s": t1 - t0, "exit_s": t3 - t2, "export_bsr_s": t4 - t3,
            "reference": "6.7-7.1 k sites/s end to end measured for the reference in the build container (SURVEY 6.2)"}


class Bench:
    """Everything one rank needs to time recursions on its GPU."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.torch, self.dist, self.args = torch, dist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            # (stdout carries the JSON line only: claim_stdout() has pointed fd 1 at stderr for NCCL's banner)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.dev = f"cuda:{self.local}"
        self.stream = torch.cuda.Stream(device=self.local)  # the library launches on this stream; events are recorded on it
        torch.cuda.set_stream(self.stream)
        self.peak, self.peak_src = measured_peak()

    # -- helpers ------------------------------------------------------------------------------
    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.cpu()]

    def build(self, cfg_key, host=None):
        import bodge_b200 as b
        from bodge_b200 import workloads

        cfg = workloads.CONFIGS[cfg_key]
        system = b.Hamiltonian(b.CubicLattice(cfg["shape"]), device=self.local)
        system.fill(*(host if host is not None else cfg["build"](cfg["shape"])))
        system._sys.set_stream(self.stream.cuda_stream)
        return system

    def timed(self, system, cols, kernel, K, W, *, col_offset=None, probe_rows=None, reduce_moments=True, scale=None):
        """W warm-up + K timed steps of `kernel`, then the single exchange of the path (summed moments of all column
        shards).  Times are the max over ranks."""
        torch, dist, s = self.torch, self.dist, system._sys
        scale = system.spectral_bound() if scale is None else scale
        if probe_rows is not None:
            s.cheb_begin(probe_rows=probe_rows, scale=scale, kernel=kernel)
        else:
            s.cheb_begin(n_random=cols, seed=1234, col_offset=self.rank * cols if col_offset is None else col_offset,
                         scale=scale, kernel=kernel)
        s.cheb_reserve(W + K + 8)
        s.cheb_steps(W)
        info, fmt = s.cheb_info(), s.cheb_format()
        launches0, avail0 = info["launches"], s.cheb_available()
        mu_dev = torch.empty(avail0 + 2 * (K + 1), dtype=torch.float64, device=self.dev)  # (+1: an odd K rounded up)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        self.barrier()
        torch.cuda.synchronize()
        e0.record(self.stream)
        s.cheb_steps(K)
        e1.record(self.stream)
        step_launches = s.cheb_info()["launches"] - launches0
        n_mom = s.cheb_available()
        if reduce_moments:
            s.cheb_read(n_mom, cols, summed=True, device_ptr=mu_dev.data_ptr())
            if self.world > 1:
                dist.all_reduce(mu_dev[:n_mom])
        e2.record(self.stream)
        torch.cuda.synchronize()
        self.barrier()
        total_ms, kernel_ms = self.max_over_ranks([e0.elapsed_time(e2), e0.elapsed_time(e1)])
        steps = (n_mom - avail0) // 2
        n_sites = system.lattice.size
        kname = fmt["kernel"]
        moved_step = fmt["matrix_bytes_per_step"] + VECTOR_PASSES.get(kname, 192) * n_sites * cols
        return {"kernel": kname, "steps": steps, "total_ms": total_ms, "kernel_ms": kernel_ms,
                "step_launches": step_launches, "gpu_launches": s.cheb_info()["launches"] - launches0,
                "ms_per_step": total_ms / steps, "kernel_ms_per_step": kernel_ms / steps,
                "steps_per_launch": steps / max(step_launches, 1), "bytes_per_step": info["bytes_per_step"],
                "moved_bytes_per_step": moved_step, "distinct_blocks": fmt["distinct_blocks"], "n_blocks": info["n_blocks"],
                "panel_width": info["panel_width"], "mu": mu_dev[:n_mom] if reduce_moments else None, "scale": scale}

    def summary(self, t, cfg_key, cols, *, jobs):
        """Compact record of a `timed()` result: throughput + the physical roofline fraction."""
        key = f"{cfg_key}_k{cols}_{t['kernel']}"
        traffic = recorded_traffic(key)  # ncu DRAM bytes per LAUNCH of the committed capture
        moved_launch = t["moved_bytes_per_step"] * t["steps_per_launch"]
        phys_launch = traffic if traffic else moved_launch
        ms_launch = t["kernel_ms"] / max(t["step_launches"], 1)
        achieved = phys_launch / (ms_launch * 1e-3) / 1e9
        alg = t["bytes_per_step"] * t["steps"] / (t["kernel_ms"] * 1e-3) / 1e9
        return {"config": cfg_key, "cols_per_gpu": cols, "kernel": t["kernel"], "steps_per_s": jobs * t["steps"] / (t["total_ms"] * 1e-3),
                "kernel_ms_per_step": t["kernel_ms_per_step"], "timed_s": t["total_ms"] * 1e-3, "timed_steps": t["steps"],
                "distinct_blocks": t["distinct_blocks"], "n_blocks": t["n_blocks"],
                "achieved_GBps": achieved, "frac": achieved / self.peak,
                "bytes_source": f"ncu dram bytes (profiles/traffic.json:{key})" if traffic else "format accounting (bdg_cheb_format)",
                "moved_bytes_per_launch": moved_launch, "steps_per_launch": t["steps_per_launch"],
                "speedup_vs_one_pass_roofline": alg / self.peak}


def incremental_update_cost(b, system, scale, n_sites):
    """SURVEY 8f-3: `fill()` of 16 / of N/2 on-site terms followed by `bdg_cheb_begin` (the first launch of the next
    recursion included), with the copies patched in place -- and, for comparison, rebuilt (BDG_NO_PATCH=1)."""
    s = system._sys
    out = {}

    def begin():
        s.cheb_begin(n_random=8, seed=1, scale=scale, kernel="auto_moments")
        s.sync()

    begin()
    for label, sites in (("16_terms", np.arange(0, n_sites, max(n_sites // 16, 1), dtype=np.int32)[:16]),
                         ("half_the_sites", np.arange(n_sites // 2, dtype=np.int32))):
        for mode in ("patched", "rebuilt"):
            if mode == "rebuilt":
                os.environ["BDG_NO_PATCH"] = "1"
            rows = []
            for rep in range(4):
                vals = np.broadcast_to((3.0 + 0.01 * rep) * b.σ0 - 0.3 * b.σ3, (len(sites), 2, 2)).astype(np.complex128).copy()
                s.sync()
                t0 = time.perf_counter()
                system.fill(sites, sites, vals)
                s.sync()
                t1 = time.perf_counter()
                begin()
                rows.append((t1 - t0, time.perf_counter() - t1))
            os.environ.pop("BDG_NO_PATCH", None)
            fill_ms, begin_ms = (1e3 * statistics.median(r[k] for r in rows[1:]) for k in (0, 1))
            out[f"{label}_{mode}"] = {"entries": int(len(sites)), "fill_ms": fill_ms, "next_recursion_begin_ms": begin_ms,
                                      "h2d_bytes": int(len(sites)) * 72}
    out["stats"] = s.stats()
    out["what"] = ("Hamiltonian.fill(on-site terms from pageable host memory: H2D + lookup + scatter + symmetry fill + Hermitian check "
                   "on the written blocks + patch of the compacted matrix / fixed-width rows / dictionary / direction codes), then "
                   "bdg_cheb_begin incl. its first launch; 'rebuilt' = the same with the copies rebuilt from scratch")
    return out


def pinned_h2d_peak(torch, local, nbytes=1 << 29):
    """Measured pinned-host -> device copy rate (GB/s): the roofline of the assembly (its inputs cross PCIe once)."""
    host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    dev = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{local}")
    best = 0.0
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        dev.copy_(host, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    return best


def dump_moments(B, system, head, cols, out_dir):
    """``--dump-outputs``: the Chebyshev moments mu_n of the headline recursion once its last timed step is done, as a
    caller of the path receives them, in float64: ``moments.npy`` [n, columns] per column (every rank's columns in rank
    order), ``moments_summed.npy`` [n] summed over all columns (what the timed region reads), ``moment_index.npy`` [n]
    the orders n.  Should the three exceed DUMP_BYTES, a fixed, seeded sample of the orders is kept, the moments of the
    last step always among them.  Collective over the ranks; rank 0 writes."""
    torch = B.torch
    n_mom = len(head["mu"])
    per_col = system._sys.cheb_read(n_mom, cols)
    if B.world > 1:
        mine = torch.from_numpy(per_col).to(B.dev)
        parts = [torch.empty_like(mine) for _ in range(B.world)]
        B.dist.all_gather(parts, mine)
        per_col = torch.cat(parts, dim=1).cpu().numpy()
    if B.rank != 0:
        return
    row_bytes = 8 * (per_col.shape[1] + 2)
    n = np.arange(n_mom)
    if n_mom * row_bytes > DUMP_BYTES - 4096:  # (4096: room for the .npy headers)
        keep = (DUMP_BYTES - 4096) // row_bytes
        n = np.concatenate([np.sort(np.random.default_rng(0).choice(n_mom - 2, keep - 2, replace=False)), n[-2:]])
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("moments", per_col[n]), ("moments_summed", head["mu"].cpu().numpy()[n]),
                      ("moment_index", n.astype(np.float64))):
        np.save(os.path.join(out_dir, f"{name}.npy"), arr)


def run_ours(args):
    import bodge_b200 as b
    from bodge_b200 import workloads

    B = Bench(args)
    torch, dist, rank, world, local = B.torch, B.dist, B.rank, B.world, B.local
    cfg = workloads.CONFIGS[args.config]
    shape, cols, K, W = cfg["shape"], args.cols, args.steps, max(args.warmup, 3)
    scaling = "weak"
    if args.total_cols > 0:
        if args.total_cols % world:
            raise SystemExit(f"--total-cols {args.total_cols} is not divisible by {world} GPUs")
        cols, scaling = args.total_cols // world, "strong"
    extras = args.config == "C5" and not args.no_extras and args.total_cols == 0

    # ---- inputs: Hamiltonian terms as packed arrays in pinned host memory --------------------
    packed = cfg["build"](shape)
    pinned = [torch.from_numpy(np.ascontiguousarray(arr)).pin_memory() for arr in packed]
    host = [t.numpy() for t in pinned]
    h2d_bytes = sum(a.nbytes for a in host)

    # ---- assembly (timed separately: the second half of BASELINE.json's metric) ---------------
    # One untimed warm-up (lazy module loading, first allocations), then the median of three full
    # assemblies: skeleton on the device, H2D of the packed Hamiltonian terms from pinned host memory,
    # scatter + symmetry fill + Hermitian check, zero-block compaction.  Everything a Hamiltonian owns
    # is released in between (bdg_destroy), so every repetition allocates its 1.3 GB again.
    def assemble_once():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sysm = b.Hamiltonian(b.CubicLattice(shape), device=local)
        sysm._sys.sync()
        t1 = time.perf_counter()
        dev = sysm.fill(*host)
        sysm._sys.sync()
        t2 = time.perf_counter()
        nfo = sysm._sys.cheb_info()  # builds the compacted BSR the Chebyshev engine consumes
        sysm._sys.sync()
        t3 = time.perf_counter()
        return sysm, dev, nfo, (t1 - t0, t2 - t1, t3 - t2)

    system, max_dev, info0, cold = assemble_once()
    reps = []
    for _ in range(3):
        del system
        system, max_dev, info0, times = assemble_once()
        reps.append(times)
    reps.sort(key=sum)
    t_skel, t_fill, t_pack = reps[1]
    n_sites = system.lattice.size
    h2d_peak = pinned_h2d_peak(torch, local)
    assembly = {
        "sites_per_s": n_sites / (t_skel + t_fill + t_pack), "unit": "sites/s", "n_sites": n_sites,
        "n_blocks": info0["n_blocks"], "skeleton_s": t_skel, "h2d_scatter_check_s": t_fill, "compaction_s": t_pack,
        "cold_first_call_s": sum(cold), "h2d_bytes": h2d_bytes, "hermitian_dev": max_dev,
        "bound": "pcie (the packed Hamiltonian terms cross host -> device once)",
        "h2d_GBps": h2d_bytes / (t_skel + t_fill + t_pack) / 1e9, "pinned_h2d_peak_GBps": h2d_peak,
        "frac": h2d_bytes / (t_skel + t_fill + t_pack) / 1e9 / h2d_peak,
        "reference_published": "7.83 k sites/s at 2^20 sites (misc/benchmark.csv:40, the reference's own benchmark model)",
        "what": "median of 3 after 1 warm-up: bdg_create_cubic + bdg_scatter (pinned host arrays -> device, symmetry "
                "fill, Hermitian check) + zero-block compaction; frac = input bytes / time against the measured pinned-copy rate",
    }
    if rank == 0:
        assembly["dict_api"] = dict_api_assembly(b, local)

    system._sys.set_stream(B.stream.cuda_stream)
    scale = system.spectral_bound()

    # ---- device-resident timing: the headline ----------------------------------------------------
    with ClockSampler(local) as clocks:
        head = B.timed(system, cols, args.kernel, K, W, scale=scale)
    mu_all = head["mu"]
    mu0 = float(mu_all[0].cpu())
    jobs = world if scaling == "weak" else 1
    assert abs(mu0 - 4.0 * n_sites * cols * world) < 1e-6 * mu0, "moment 0 must equal the number of vector entries"
    mu16 = mu_all[:16].cpu().numpy().copy()
    if args.dump_outputs:
        dump_moments(B, system, head, cols, args.dump_outputs)

    # ---- parity at N > 1: every shard's columns recomputed on rank 0 ----------------------------------
    parity = None
    if world > 1:
        ok = torch.zeros(1, dtype=torch.float64, device=B.dev)
        if rank == 0:
            s = system._sys
            s.cheb_begin(n_random=cols * world, seed=1234, col_offset=0, scale=scale, kernel=args.kernel)
            s.cheb_steps(max(0, 7 - (s.cheb_available() // 2 - 1)))
            alone = s.cheb_read(16, cols * world, summed=True)
            err = float(np.max(np.abs(alone - mu16)) / np.max(np.abs(mu16)))
            parity = {"what": f"first 16 summed moments of all {cols * world} columns: all-reduce over {world} column shards vs "
                              "one GPU computing every column", "max_rel_err": err, "tolerance": 1e-12, "ok": bool(err <= 1e-12)}
            ok[0] = 1.0 if err <= 1e-12 else 0.0
        dist.broadcast(ok, 0)
        assert float(ok.cpu()) == 1.0, "sharded moments differ from the single-GPU recomputation"

    # ---- comparison runs on the same matrix ----------------------------------------------------------
    plain = three_term = None
    if not args.no_plain and head["kernel"] != "ell":
        try:
            t = B.timed(system, cols, "ell", K, W, scale=scale)
            plain = B.summary(t, args.config, cols, jobs=jobs)
        except (ValueError, RuntimeError):
            plain = None
    if not args.no_plain and head["kernel"] == "t2":
        # the literal three-term recursion (every T_n materialised): two steps per launch and one step per launch
        three_term = {}
        for name in ("pair", "dict_diag"):
            try:
                t = B.timed(system, cols, name, K, W, scale=scale)
            except (ValueError, RuntimeError):
                continue
            three_term[t["kernel"]] = B.summary(t, args.config, cols, jobs=jobs)

    # ---- strong scaling: 64 columns in total (SURVEY 8e "report both") ----------------------------------
    strong = None
    if extras and 64 % world == 0:
        kc = 64 // world
        t = B.timed(system, kc, args.kernel, K, W, col_offset=rank * kc, scale=scale)
        strong = B.summary(t, args.config, kc, jobs=1)
        strong["total_cols"] = 64
        strong["what"] = "one job of 64 columns split over the GPUs: steps/s of the whole job (a step is done when every shard has done it)"

    # ---- end to end through the public API with host buffers -------------------------------------
    e2e = None
    if not args.no_e2e:
        system._sys.set_stream(None)
        e2e_steps = 1024  # 2050 moments: the recursion length of the C5 free-energy evaluation
        calls = 2

        def one_call():
            system.fill(*host)  # H2D of all Hamiltonian terms + scatter + Hermitian check
            return system.chebyshev_moments(2 * e2e_steps + 2, vectors=cols * world, seed=1234, summed=True, kernel=args.kernel)

        one_call()
        B.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(calls):
            mu = one_call()
        torch.cuda.synchronize()
        B.barrier()
        dt = B.max_over_ranks([time.perf_counter() - t0])[0]
        e2e = {"value": jobs * calls * e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": h2d_bytes / e2e_steps, "d2h_bytes_per_step": mu.nbytes / e2e_steps,
               "what": f"{calls} x [Hamiltonian.fill(pinned host arrays) + chebyshev_moments({2 * e2e_steps + 2}) -> host]; "
                       f"{e2e_steps} steps per call", "seconds": dt}
        system._sys.set_stream(B.stream.cuda_stream)

    # ---- the reference's parameter-sweep idiom: re-enter `with` for some on-site terms, start the next recursion -------
    incremental = None
    if extras and rank == 0:
        incremental = incremental_update_cost(b, system, scale, n_sites)
    del system

    # ---- less block repetition on the same lattice; the other BASELINE configs ----------------------
    repetition = others = None
    if extras:
        repetition = {}
        for key in ("C5_disordered", "C5_random", "C5_periodic"):
            try:
                sysx = B.build(key)
                t = B.timed(sysx, cols, args.kernel, K, W)
                repetition[key] = B.summary(t, key, cols, jobs=jobs)
                repetition[key]["workload"] = workloads.CONFIGS[key]["label"]
                del sysx
            except (RuntimeError, ValueError, MemoryError) as err:  # an extra must not take the headline down with it
                repetition[key] = {"error": str(err)[:200]}
        others = {}
        # C2: 256 stochastic columns per GPU; C4: 8 per GPU; C3: 1024 probe sites x 4 components, sharded (strong)
        for key, kc in (("C2", 256), ("C4", 8)):
            try:
                sysx = B.build(key)
                t = B.timed(sysx, kc, args.kernel, K, W)
                others[key] = B.summary(t, key, kc, jobs=jobs)
                if key == "C4" and others[key]["kernel"] == "t2":
                    # three-dimensional lattice: the even-vector kernel (csrc/cheb_cube.cu) moves half the bytes in about the
                    # time of the single-step kernel -- both, so that steps/s and the roofline fraction can be read side by side
                    t1 = B.timed(sysx, kc, "dict_diag", K, W)
                    others["C4_single_step"] = B.summary(t1, key, kc, jobs=jobs)
                del sysx
            except (RuntimeError, ValueError, MemoryError) as err:
                others[key] = {"error": str(err)[:200]}
        sysx = B.build("C3")
        sites = [(3 * p + 2, 3 * q + 2, 0) for p in range(32) for q in range(32)]
        rows = sysx._probe_rows(sites)
        lo, hi = b.distributed.shard_range(len(rows), rank, world)
        t = B.timed(sysx, hi - lo, args.kernel, K, W, probe_rows=rows[lo:hi], reduce_moments=False)
        others["C3"] = B.summary(t, "C3", hi - lo, jobs=1)
        others["C3"]["what"] = "4096 probe columns (1024 sites x 4) sharded over the GPUs: steps/s of the whole LDOS job"
        if world == 1:  # BASELINE shards C3 over 2/4/8 GPUs: one GPU's share of the 8-GPU run (512 columns) beside the whole job
            t8 = B.timed(sysx, 512, args.kernel, K, W, probe_rows=rows[:512], reduce_moments=False)
            others["C3_share_of_8"] = B.summary(t8, "C3", 512, jobs=1)
            others["C3_share_of_8"]["what"] = "the 512 probe columns one GPU holds when C3 is sharded over 8 GPUs (SURVEY 8d)"
        # the exchange of this path: all-gather of the per-column moments (column order = rank order), checked
        if world > 1:
            mine = torch.from_numpy(sysx._sys.cheb_read(8, hi - lo)).to(B.dev)
            parts = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(parts, mine)
            if rank == 0:
                s = sysx._sys
                probe = np.concatenate([rows[b.distributed.shard_range(len(rows), r, world)[0]:][:8] for r in range(world)])
                s.cheb_begin(probe_rows=probe, scale=t["scale"], kernel=args.kernel)
                s.cheb_steps(max(0, 3 - (s.cheb_available() // 2 - 1)))
                want = s.cheb_read(8, len(probe))
                got = np.concatenate([p.cpu().numpy()[:, :8] for p in parts], axis=1)
                err = float(np.max(np.abs(got - want)))
                others["C3"]["gather_check"] = {"what": "first 8 moments of the first 8 columns of every shard after the all-gather "
                                                        "vs one GPU computing those columns", "max_abs_err": err, "ok": bool(err <= 1e-12)}
        del sysx

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ------------------------------------------------------------
    hs = B.summary(head, args.config, cols, jobs=jobs)
    roofline = {"bound": "hbm", "achieved": hs["achieved_GBps"], "peak": B.peak, "unit": "GB/s", "frac": hs["frac"],
                "traffic": recorded_traffic(f"{args.config}_k{cols}_{head['kernel']}"), "peak_source": B.peak_src,
                "bytes_source": hs["bytes_source"],
                "kernel": KERNEL_NAMES.get(head["kernel"], head["kernel"]), "steps_per_launch": head["steps_per_launch"],
                "kernel_ms_per_launch": head["kernel_ms"] / max(head["step_launches"], 1), "matrix_format": head["kernel"],
                "distinct_blocks": head["distinct_blocks"], "moved_bytes_per_launch": hs["moved_bytes_per_launch"],
                "algorithmic_bytes_per_launch": head["bytes_per_step"] * head["steps_per_launch"],
                "speedup_vs_one_pass_roofline": hs["speedup_vs_one_pass_roofline"],
                "note": "frac = bytes the kernel moves per launch / its CUDA-event time / the measured copy peak.  The SURVEY-8d "
                        "algorithmic bytes (every 4x4 block + index + three vector passes per step) over the same time give "
                        "speedup_vs_one_pass_roofline: > 1 because the block dictionary takes the matrix out of the stream and the "
                        "even-vector recursion moves three vector passes per TWO steps",
                "assembly": assembly}
    if three_term:
        roofline["three_term_recursion"] = three_term
    if plain is not None:
        roofline["plain"] = plain

    cpu = None
    if not args.no_cpu_baseline:
        res = cpu_chebyshev(args.config, cols, steps=3, warmup=1, budget_s=20.0, moments_for_parity=16 if world == 1 else 0)
        cpu = {"value": 1e3 / res["ms_per_step"], "unit": UNIT, "cores": res["cores"], "kind": "port",
               "sample": f"3 steps after 1 warm-up of the same workload (k={cols}) on {res['fraction']:.3f} of the block rows, "
                         f"scipy bsr_matvecs, rows split over {res['cores']} processes; numpy assembly took {res['assembly_s']:.1f} s",
               "assembly_sites_per_s": res["n_sites"] / res["assembly_s"]}
        if world == 1:
            want = res["moments"].sum(axis=1)
            err = float(np.max(np.abs(want - mu16)) / np.max(np.abs(want)))
            parity = {"what": f"first 16 summed moments of the {cols} timed columns vs the CPU oracle (scipy three-term recursion on the "
                              f"oracle-assembled matrix, {res['moments_s']:.1f} s)", "max_rel_err": err, "tolerance": 1e-10,
                      "ok": bool(err <= 1e-10)}
            assert parity["ok"], f"GPU moments differ from the CPU oracle by {err:.3e}"

    line = {
        # weak scaling: every GPU advances its own 8-column job, the job count adds up; strong scaling:
        # one job of --total-cols columns, a step is done when every shard has done it
        "metric": METRIC, "value": jobs * head["steps"] / (head["total_ms"] * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
        "warmup": W, "timed_steps": head["steps"], "timed_s": head["total_ms"] * 1e-3,
        "ms_per_step": head["total_ms"] / head["steps"], "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.config, cfg, n_sites, head["n_blocks"], cols),
        "run": {"parallelism": f"column shards x{world}, matrix replicated", "kernel": head["kernel"], "panel_width": head["panel_width"],
                "recursion": ("even-vector form E_{j+1} = 2 T_2(H~) E_j - E_{j-1} (two steps per launch)" if head["kernel"] == "t2"
                              else "three-term T_{n+1} = 2 H~ T_n - T_{n-1}")},
        "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": head["gpu_launches"], "roofline": roofline,
        "parity_check": parity, "cpu_baseline": cpu, "block_repetition": repetition, "other_configs": others,
        "strong_scaling": strong, "incremental_update": incremental,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to
    fd 1 when it creates a communicator), so keep a private duplicate of the real stdout for the JSON line and
    point fd 1 at stderr for everything else.  NCCL_DEBUG is left as the caller set it."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    args = parse_args()
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
