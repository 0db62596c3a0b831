#!/usr/bin/env python
"""bench.py - "assembled DoFs/s + CG solve s (SWIPDG p1, 16M cells)" on N B200s of one node.

A step is one pass of the hot path over the workload: assemble every affine part of the system matrix and of the rhs
(K2 + K3), then freeze and CG-solve to ||r||/||b|| <= 1e-10 (K4 - K6), on the 4096^2 structured Q1 grid with ESV2007 data
(BASELINE.json configs[4], the configuration the metric is quoted on; --grid scales it down for a quick look).

    value          assembled DoFs/s over all ranks: K * N_dofs / sum of the K assembly times (device time, max over ranks)
    cg_solve_s     mean CG time-to-solution of the K steps (device time), with cg_iterations and cg_s_per_iteration;
                   default solver "cg.mg" (CG with the two-level multigrid preconditioner); cg_diagonal holds the plain
                   Jacobi-CG solve of the same system, run once after the timed steps
    ms_per_step    whole step (assembly + solve), wall clock between barriers / K
    e2e            the same through the public API from HOST buffers: grid arrays -> hdd_mesh_create (H2D) -> init -> solve
                   -> solution back on the host (D2H), every step
    roofline       the dominant kernel (CG SpMV with fused p.Ap): algorithmic bytes / CUDA-event time / measured HBM peak
    cpu_baseline   the CPU oracle (a port: the reference cannot be built here) on a bounded sample, rank 0, N = 1 only

`--impl reference` times the CPU restatement of the reference path (oracle/, serial walk like the reference) instead.
`--dump-outputs DIR` writes what the last timed step computed (solution, system matrix, rhs; see dump_outputs) as .npy
files: the inputs are the same for the same arguments, so two builds can be compared output for output.
N > 1: one rank per GPU (torchrun); the 8 x 8 subdomains of BlockSWIPDG are dealt to the ranks in contiguous slabs,
NCCL carries the coupling-face halo of the CG direction and the dot-product all-reduces (strong scaling of one grid).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "assembled DoFs/s + CG solve s (SWIPDG p1, 16M cells)"
PRECISION = 1e-10


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """samples SM clocks and throttle reasons during the timed region: through NVML in-process (no fork, no driver
    re-initialisation next to a launch-bound step), falling back to spawning nvidia-smi"""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self._halt, self._was_started = index, [], threading.Event(), False
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK -> physical device: respect CUDA_VISIBLE_DEVICES when it lists plain indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    phys = int(ids[index])
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        sm = n.nvmlDeviceGetClockInfo(self._handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self._handle, n.NVML_CLOCK_SM)
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        r = get(self._handle)
        bits = [getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8), getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20), getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)]
        return [str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b in bits]

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        return [x.strip() for x in out.strip().split(",")]

    def start(self):
        self._was_started = True
        super().start()

    def run(self):
        while not self._halt.is_set():
            try:
                f = self._sample_nvml() if self._nvml else self._sample_smi()
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            self._halt.wait(0.05 if self._nvml else 0.2)

    def stop(self):
        self._halt.set()
        if self._was_started:
            self.join(timeout=3)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        reasons = [n for k, n in enumerate(self.NAMES) if any(s[2 + k].lower().startswith("active") for s in self.samples)]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples), "source": "nvml" if self._nvml else "nvidia-smi"}


def workload_config(n, solver, world):
    """the `config` object of both arms (identical for identical arguments)"""
    return {"workload": "config5: SWIPDG p1 (Q1) on the %dx%d structured grid [-1,1]^2, ESV2007 data, 8x8 BlockSWIPDG "
                        "partition" % (n, n), "cells": n * n, "dofs": 4 * n * n,
            "cg": "%s to ||r||/||b|| <= 1e-10" % solver,
            "l2_flush": "inputs >> L2 (matrix %.1f GB per part)" % (8.0 * 16 * (n * n + 2 * 2 * n * (n - 1)) / 1e9),
            "parallelism": "subdomain slabs x%d" % world}


class CpuWorkload:
    """the oracle (CPU port of the reference) on an n x n sample of the workload: mesh + pattern once, then per step the
    assembly walk and `cg_iters` Jacobi-CG iterations"""

    def __init__(self, n):
        from oracle import oracle as o
        self.o, self.n = o, n
        self.m = o.mesh_cube(n, n, -1.0, 1.0, -1.0, 1.0)
        t0 = time.perf_counter()
        self.rp, self.col = o.pattern(self.m)
        self.t_pattern = time.perf_counter() - t0

    def step(self, threads, cg_iters):
        o = self.o
        o.set_threads(threads)
        try:
            t0 = time.perf_counter()
            A = o.assemble_lhs(self.m, o.const(1.0), None, self.rp, self.col)
            b = o.assemble_rhs(self.m, o.esv2007_force())
            t_asm = time.perf_counter() - t0
            t0 = time.perf_counter()
            x, it, rr = o.cg(self.rp, self.col, A, b, precond=1, rtol=1e-30, maxit=cg_iters)
            t_cg = time.perf_counter() - t0
        finally:
            o.set_threads(1)
        return t_asm, t_cg / max(it, 1), it

    def solve(self, threads, rtol=PRECISION):
        """Jacobi-CG to the bench's precision (the "CG solve s" half of the metric on this sample)"""
        o = self.o
        o.set_threads(threads)
        try:
            A = o.assemble_lhs(self.m, o.const(1.0), None, self.rp, self.col)
            b = o.assemble_rhs(self.m, o.esv2007_force())
            t0 = time.perf_counter()
            x, it, rr = o.cg(self.rp, self.col, A, b, precond=1, rtol=rtol, maxit=200000)
            return time.perf_counter() - t0, it, rr
        finally:
            o.set_threads(1)

    def record(self, step, threads, cg_iters):
        t_asm, t_it, it = step
        n = self.n
        return {"value": self.m.n_dofs / t_asm, "unit": "DoFs/s", "cores": threads, "kind": "port",
                "sample": "%dx%d Q1 cells (ESV2007 data): assembly walk + %d Jacobi-CG iterations, %d host thread%s"
                          % (n, n, it, threads, "" if threads == 1 else "s"),
                "assemble_s": t_asm, "pattern_s": self.t_pattern, "cg_s_per_iteration": t_it,
                "note": "CPU restatement of the reference (oracle/); the reference itself needs un-vendored DUNE modules"}


def cpu_estimator_sample(squares=256):
    """the oracle's four estimator walks (one function) on 8 * squares^2 triangles, one core -> (cells, seconds)"""
    from oracle import oracle as o
    m = o.mesh_bisect(squares, -1.0, 1.0, 2)
    v = m.xy[m.cv]
    u = (np.cos(0.5 * np.pi * v[..., 0]) * np.cos(0.5 * np.pi * v[..., 1])).reshape(-1)
    t0 = time.perf_counter()
    o.indicators(m, u, o.esv2007_force(), o.const(1.0))
    return m.nc, time.perf_counter() - t0


def cpu_baseline(n_cpu, cg_iters, solve_n):
    """oracle (port of the reference's serial walk) on a bounded sample: n_cpu^2 Q1 cells, cg_iters CG iterations.
    `value` is the faithful one-core number (the reference's walk is serial, discretizations/swipdg.hh:485); all_cores
    repeats the sample with the oracle's optional host threading (SURVEY 8d asks for both); `solve` is a Jacobi-CG solve
    to 1e-10 on solve_n^2 cells with all threads, `estimator` the oracle's estimator walks on 524288 triangles."""
    w = CpuWorkload(n_cpu)
    out = w.record(w.step(1, cg_iters), 1, cg_iters)
    cores = os.cpu_count() or 1
    rec = w.record(w.step(cores, cg_iters), cores, cg_iters)
    out["all_cores"] = {"cores": cores, "value": rec["value"], "assemble_s": rec["assemble_s"],
                        "cg_s_per_iteration": rec["cg_s_per_iteration"],
                        "note": "same sample with the oracle's own threading (atomic scatter); the reference has none"}
    ws = w if solve_n == n_cpu else CpuWorkload(solve_n)
    t, it, rr = ws.solve(cores)
    out["solve"] = {"grid": "%dx%d" % (solve_n, solve_n), "solver": "cg.diagonal", "cores": cores, "seconds": t,
                    "iterations": it, "relative_residual": rr}
    cells, te = cpu_estimator_sample()
    out["estimator"] = {"triangles": cells, "seconds": te, "cells_per_s": cells / te, "cores": 1,
                        "sample": "ESV2007 indicators (Oswald, P0 f, RT0 flux, eta_NC / eta_R / eta_DF) on %d triangles" % cells}
    return out


def default_cpu_n(n):
    """the CPU arm runs the bench's own grid when the host has the memory for the oracle's CSR arrays (~1.3 KB per cell),
    else the largest power-of-two fraction of it that fits"""
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 32 << 30
    m = n
    while m > 256 and 1400.0 * m * m > 0.6 * avail:
        m //= 2
    return m


def run_reference(args):
    """The CPU arm: the oracle port with all the host threads it can use (its own threading; the reference's walk is
    serial, the one-core figure is reported next to it), on the bench's own grid."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_cpu = args.cpu_n if args.cpu_n > 0 else default_cpu_n(args.n)
    cores = os.cpu_count() or 1
    w = CpuWorkload(n_cpu)
    steps = []
    for k in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        rec = w.record(w.step(cores, args.cpu_cg_iters), cores, args.cpu_cg_iters)
        steps.append((time.perf_counter() - t0, rec))
    timed = steps[args.warmup:]
    cb = timed[-1][1]
    value = float(np.mean([s[1]["value"] for s in timed]))
    cb["value"] = value
    # outside the timed steps: the same walk on one core (bounded: a 1024^2 sample when the grid is larger) and a
    # Jacobi-CG solve to 1e-10 on a 768^2 sample with all threads
    n_one = min(n_cpu, 1024)
    w1 = w if n_one == n_cpu else CpuWorkload(n_one)
    one = w1.record(w1.step(1, min(args.cpu_cg_iters, 5)), 1, args.cpu_cg_iters)
    cb["one_core"] = {"cores": 1, "value": one["value"], "assemble_s": one["assemble_s"], "grid": "%dx%d" % (n_one, n_one),
                      "cg_s_per_iteration": one["cg_s_per_iteration"],
                      "note": "the walk as the reference runs it: serial (discretizations/swipdg.hh:485)"}
    ws = CpuWorkload(args.cpu_solve_n) if args.cpu_solve_n != n_cpu else w
    t, it, rr = ws.solve(cores)
    cb["solve"] = {"grid": "%dx%d" % (args.cpu_solve_n, args.cpu_solve_n), "solver": "cg.diagonal", "cores": cores,
                   "seconds": t, "iterations": it, "relative_residual": rr}
    config = workload_config(args.n, args.solver, args.gpus)
    if n_cpu != args.n:
        config["cpu_sample"] = "%dx%d cells (host memory)" % (n_cpu, n_cpu)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "DoFs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean([s[0] for s in timed])),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "cg_s_per_iteration": float(np.mean([s[1]["cg_s_per_iteration"] for s in timed])),
            "cpu_baseline": cb,
            "e2e": {"value": value, "unit": "DoFs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def gather_concat(local, world, torch):
    """every rank's numpy array, concatenated in rank order, on every rank (NCCL all_gather of padded device tensors)"""
    if world == 1:
        return np.asarray(local)
    import torch.distributed as dist
    local = np.ascontiguousarray(local)
    n = torch.tensor([local.shape[0]], dtype=torch.int64, device="cuda")
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n)
    sizes = [int(x.item()) for x in sizes]
    t = torch.zeros(max(sizes), dtype=torch.from_numpy(local[:0]).dtype, device="cuda")
    t[:local.shape[0]] = torch.from_numpy(local).cuda()
    parts = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(parts, t)
    return np.concatenate([p[:k].cpu().numpy() for p, k in zip(parts, sizes)])


DUMP_SAMPLE = 1 << 21  # entries per dumped array: three arrays of float64 stay under 64 MB


class _DeviceArray:
    """a float64 device buffer of the library, for torch to view without a copy"""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3,
                                         "strides": None}


def dump_outputs(dirname, d, torch, capi, rank, world):
    """What the last timed step leaves its caller - the solution of the solve, the CSR values (over pattern()) of the
    assembled system matrix and the assembled rhs - as <dirname>/{solution,system_matrix,rhs}.npy in float64.  A longer
    array than DUMP_SAMPLE entries is sampled at the sorted global indices numpy.random.default_rng(0) draws without
    replacement, so that runs with the same arguments write the same entries.  Collective on N > 1 ranks (rank order is
    global order); rank 0 writes."""
    import ctypes as C
    x = C.c_void_p()
    capi.check(capi.lib().hdd_solution_dev(d._h, C.byref(x)))
    arrays = {"solution": (x.value, d.num_owned_dofs()), "system_matrix": d.system_matrix().device_pointer(-1),
              "rhs": d.rhs().device_pointer(-1)}
    if rank == 0:
        os.makedirs(dirname, exist_ok=True)
    for name, (ptr, n) in arrays.items():
        counts = gather_concat(np.array([n], np.int64), world, torch)
        total, offset = int(counts.sum()), int(counts[:rank].sum())
        if total <= DUMP_SAMPLE:
            idx = np.arange(total)
        else:
            idx = np.sort(np.random.default_rng(0).choice(total, DUMP_SAMPLE, replace=False))
        mine = torch.from_numpy(idx[(idx >= offset) & (idx < offset + n)] - offset).cuda()
        values = torch.as_tensor(_DeviceArray(ptr, n), device="cuda")[mine].cpu().numpy()
        values = gather_concat(values, world, torch)
        if rank == 0:
            np.save(os.path.join(dirname, name + ".npy"), values.astype(np.float64))


def small_grid_parity(hdd, torch, comm, rank, world, local_rank):
    """In-run parity of what this process group computes, against the CPU oracle (checker only, rank 0): a 256^2 Q1 grid
    (pattern bit-exact, entries and rhs 1e-12, cg.mg solution 1e-8) and 8192 triangles (block-Jacobi CG solution and every
    per-cell indicator 1e-8, eta_ESV2007 against the reference's golden 4.85e-02), sharded over the ranks like the
    timed workload."""
    from oracle import oracle as o
    out = {}
    # ---- Q1, the bench configuration in small -------------------------------------------------------------------
    n = 256
    g = hdd.grids.cube(n, partitions=(8, 8))
    roff = hdd.parallel.rank_cell_offsets(g, world)
    d = hdd.BlockSWIPDG(g, hdd.problems.ESV2007(), device=local_rank, cell_range=(int(roff[rank]), int(roff[rank + 1])), comm=comm)
    d.init()
    rp, col = d.pattern()
    counts = gather_concat(np.diff(rp), world, torch)
    col = gather_concat(col, world, torch)
    A = gather_concat(d.system_matrix().affine_part(), world, torch)
    b = gather_concat(d.rhs().affine_part(), world, torch)
    u, info = d.uncached_solve({"type": "cg.mg", "precision": 1e-12, "max_iter": 2000}, return_info=True)
    res = d.residual()
    u = gather_concat(u, world, torch)
    # the Jacobi solve takes the peer-memory SpMV on N > 1 ranks (halo read over NVLink inside the kernel)
    uj, info_j = d.uncached_solve({"type": "cg.diagonal", "precision": 1e-12, "max_iter": 20000}, return_info=True)
    uj = gather_concat(uj, world, torch)
    if rank == 0:
        m = o.Mesh(o.CUBE, g.xy, g.cell_verts, g.cell_neigh)
        rp_o, col_o = o.pattern(m)
        A_o = o.assemble_lhs(m, o.const(1.0), None, rp_o, col_o)
        b_o = o.assemble_rhs(m, o.esv2007_force())
        rp_g = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        # the oracle's own solution, reached by its CG from the device solution (a wrong one would neither be close nor cheap)
        u_o, it_o, rr_o = o.cg(rp_o, col_o, A_o, b_o, precond=1, rtol=1e-13, maxit=20000, x0=u)
        out["q1_256"] = {"pattern_equal": bool(np.array_equal(rp_g, rp_o) and np.array_equal(col, col_o)),
                         "entries_rel": float(np.abs(A - A_o).max() / np.abs(A_o).max()),
                         "rhs_rel": float(np.abs(b - b_o).max() / np.abs(b_o).max()),
                         "solution_rel": float(np.abs(u - u_o).max() / np.abs(u_o).max()),
                         "oracle_polish_iterations": int(it_o), "cg_mg_iterations": info["iterations"],
                         "true_residual": res, "jacobi_solution_rel": float(np.abs(uj - u_o).max() / np.abs(u_o).max()),
                         "jacobi_iterations": info_j["iterations"], "jacobi_peer_memory": bool(info_j.get("peer_memory"))}
    del d
    # ---- P1 on 8192 triangles: solve + estimators ------------------------------------------------------------------
    g = hdd.grids.simplex(32, partitions=(8, 8))
    roff = hdd.parallel.rank_cell_offsets(g, world)
    d = hdd.BlockSWIPDG(g, hdd.problems.ESV2007(), device=local_rank, cell_range=(int(roff[rank]), int(roff[rank + 1])), comm=comm)
    d.init()
    A = gather_concat(d.system_matrix().affine_part(), world, torch)
    u_loc = d.uncached_solve({"type": "cg.blockdiagonal", "precision": 1e-13, "max_iter": 20000})
    ind = d.indicators(u_loc)
    eta = d.estimate(u_loc, "eta_ESV2007")
    u = gather_concat(u_loc, world, torch)
    ind = {k: gather_concat(v, world, torch) for k, v in ind.items()}
    if rank == 0:
        m = o.Mesh(o.SIMPLEX, g.xy, g.cell_verts, g.cell_neigh)
        rp_o, col_o = o.pattern(m)
        A_o = o.assemble_lhs(m, o.const(1.0), None, rp_o, col_o)
        b_o = o.assemble_rhs(m, o.esv2007_force())
        u_o, it_o, rr_o = o.cg(rp_o, col_o, A_o, b_o, precond=1, rtol=1e-14, maxit=20000, x0=u)
        ind_o = o.indicators(m, u, o.esv2007_force(), o.const(1.0))
        worst = max(float(np.abs(ind[k] - ind_o[k]).max() / max(np.abs(ind_o[k]).max(), 1e-300))
                    for k in ("nc2", "res2", "r2", "df2", "dfstar2", "rstar2", "amin", "resstar2"))
        out["p1_8192"] = {"entries_rel": float(np.abs(A - A_o).max() / np.abs(A_o).max()),
                          "solution_rel": float(np.abs(u - u_o).max() / np.abs(u_o).max()),
                          "indicators_rel": worst, "eta_ESV2007": eta, "eta_ESV2007_golden": 4.85e-02}
    del d
    ok = True
    if rank == 0:
        q, t = out["q1_256"], out["p1_8192"]
        ok = (q["pattern_equal"] and q["entries_rel"] <= 1e-12 and q["rhs_rel"] <= 1e-12 and q["solution_rel"] <= 1e-8
              and q["jacobi_solution_rel"] <= 1e-8 and t["entries_rel"] <= 1e-12 and t["solution_rel"] <= 1e-8 and t["indicators_rel"] <= 1e-8
              and abs(t["eta_ESV2007"] - 4.85e-02) <= 0.006 * 4.85e-02)
        out["ok"] = bool(ok)
    return out, ok


def estimator_phase(hdd, torch, capi, comm, rank, world, local_rank, n, peak, peak_kind, barrier):
    """BASELINE config 4 at scale, the whole pipeline on triangles: block-SWIPDG P1 on 8 s^2 triangles of the ALU ladder
    (s = 1408 for the 4096^2-sized job: 15.9 M triangles, 47.6 M DoFs) with the 8 x 8 subdomain partition sharded over the
    ranks: assembly, cg.mg solve to 1e-10, and the a-posteriori estimator (north_star item 3) on that solution - eta_ESV2007
    through the public API from a host vector (H2D of the vector inside the timed region) and its device part alone (CUDA
    events).  Checked in the run: true residual, L2 / H1 error against the exact solution and the effectivity against the
    asymptotics of the reference's committed ladder (test/linearelliptic-swipdg-expectations_esv2007_2daluconform.cxx:32-57)."""
    import ctypes as C
    L = capi.lib()
    s = max(8, int(round(n * 1408 / 4096 / 8.0)) * 8)
    t0 = time.perf_counter()
    g = hdd.grids.simplex(s, partitions=(8, 8))
    t_grid = time.perf_counter() - t0
    roff = hdd.parallel.rank_cell_offsets(g, world)
    cr = (int(roff[rank]), int(roff[rank + 1]))
    t0 = time.perf_counter()
    d = hdd.BlockSWIPDG(g, hdd.problems.ESV2007(), device=local_rank, cell_range=cr, comm=comm)
    d.init()
    t_setup = time.perf_counter() - t0
    t_asm = min(d.assemble() for _ in range(3))
    opts = {"type": "cg.mg", "precision": PRECISION, "max_iter": 2000}
    try:
        infos = [d.uncached_solve(opts, return_info=True, copy_to_host=False)[1] for _ in range(4)]
        info = sorted(infos[1:], key=lambda i: i["seconds"])[1]  # one warm-up, then the median of three
        solver = "cg.mg"
    except hdd.discretizations.requirements_not_met:  # lattice cannot be coarsened far enough: block-Jacobi CG
        opts["type"] = solver = "cg.blockdiagonal"
        opts["max_iter"] = 200000
        _, info = d.uncached_solve(opts, return_info=True, copy_to_host=False)
    res, floor = d.residual(with_floor=True)
    norms = d.error_norms(*hdd.problems.ESV2007_EXACT, order=5)
    u = capi.pinned_empty((3 * (cr[1] - cr[0]),), np.float64)
    d.uncached_solve(opts, copy_to_host=True, out=u)
    eta = d.estimate(u, "eta_ESV2007")  # warm-up (allocations)
    barrier()
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        eta = d.estimate(u, "eta_ESV2007")
    barrier()
    t_e2e = (time.perf_counter() - t0) / reps
    e_nc, e_r, e_df = (d.estimate(u, t) for t in ("eta_NC_ESV2007", "eta_R_ESV2007", "eta_DF_ESV2007"))
    roofs = {}
    for which, name in ((4, "estimator_pass"), (5, "indicators"), (3, "assembly_p1")):
        sec, byt = C.c_double(), C.c_double()
        capi.check(L.hdd_profile_kernel(d._h, which, 5, C.byref(sec)))
        capi.check(L.hdd_kernel_bytes(d._h, which, C.byref(byt)))
        roofs[name] = {"bound": "hbm", "achieved": byt.value / sec.value / 1e9, "peak": peak, "unit": "GB/s",
                       "frac": byt.value / sec.value / 1e9 / peak, "traffic": None, "ms": sec.value * 1e3,
                       "algorithmic_bytes": byt.value, "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)"}
    try:  # DRAM traffic of the indicator kernel from the committed ncu capture of this workload on one GPU
        with open(os.path.join(ROOT, "profiles", "r02_ncu_estimator.json")) as f:
            for kk in json.load(f)["kernels"]:
                if "k_indicators" in kk["kernel"] and world == 1 and n == 4096:
                    roofs["indicators"]["traffic"] = kk["dram_bytes"] * (8 * s * s) / 16773632.0
    except Exception:
        pass
    stats = torch.tensor([t_asm, t_e2e, roofs["estimator_pass"]["ms"], info["seconds"]], dtype=torch.float64, device="cuda")
    if world > 1:
        torch.distributed.all_reduce(stats, op=torch.distributed.ReduceOp.MAX)
    t_asm, t_e2e, ms_dev, t_solve = [float(x) for x in stats.cpu()]
    n_cells, n_dofs = g.n_cells, 3 * g.n_cells
    # asymptotics of the committed ladder: L2 s^2 = 0.293, 0.290, 0.287, 0.285 -> 0.282; H1 s = 1.312, 1.296, 1.286, 1.283
    # -> 1.280; effectivity eta / energy 1.37, 1.28, 1.23, 1.21 -> 1.19; eta_R s^2 -> 1.165
    exp_l2, exp_h1, exp_r = 0.2822 / (s * s), 1.2804 / s, 1.165 / (s * s)
    eff = eta / norms["energy"]
    ok = (res <= max(1e-9, 0.25 * floor) and np.isfinite(eta) and
          (s < 64 or (abs(norms["L2"] - exp_l2) <= 0.03 * exp_l2 and abs(norms["H1_semi"] - exp_h1) <= 0.01 * exp_h1 and
                      1.15 <= eff <= 1.25 and abs(e_r - exp_r) <= 0.02 * exp_r)))
    out = {"workload": "config4 at scale: BlockSWIPDG p1 on %d triangles (ALU-ladder grid, %d^2 squares of 8), 8x8 subdomains"
                       % (n_cells, s), "triangles": n_cells, "dofs": n_dofs,
           "assemble_ms": 1e3 * t_asm, "assembled_dofs_per_s": n_dofs / t_asm,
           "solver": solver, "cg_solve_s": t_solve, "cg_iterations": info["iterations"],
           "true_residual": res, "true_residual_fp64_floor": floor,
           "L2_error": norms["L2"], "H1_semi_error": norms["H1_semi"], "L2_expected": exp_l2, "H1_semi_expected": exp_h1,
           "estimate_ms": ms_dev, "cells_per_s": n_cells / (1e-3 * ms_dev),
           "estimate_e2e_ms": 1e3 * t_e2e, "e2e_h2d_bytes": int(8 * n_dofs),
           "eta_ESV2007": eta, "eta_NC": e_nc, "eta_R": e_r, "eta_DF": e_df, "effectivity": eff, "eta_R_expected": exp_r,
           "ok": bool(ok),
           "roofline_estimator": roofs["estimator_pass"], "roofline_indicators": roofs["indicators"],
           "roofline_assembly_p1": roofs["assembly_p1"], "grid_generation_s": t_grid, "create_init_s": t_setup,
           "note": "estimate_ms is the device part (Oswald + indicator kernel + reductions, CUDA events), estimate_e2e_ms the "
                   "public call from a page-locked host vector; the indicator kernel is bound by the fp64 pipe (32 force "
                   "evaluations per triangle prescribed by the reference's quadrature orders), not by HBM"}
    del d
    return out, bool(ok)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--grid", dest="n", type=int, default=4096, help="cells per side of the structured grid")
    ap.add_argument("--cpu-n", type=int, default=0, help="CPU sample: cells per side (0: reference arm = --grid if the host "
                                                         "memory allows, cpu_baseline of the GPU arm = 768)")
    ap.add_argument("--cpu-cg-iters", type=int, default=0, help="0: 100 * (768 / cpu_n)^2, at least 3")
    ap.add_argument("--cpu-solve-n", type=int, default=768)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-estimator", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the small-grid check against the CPU oracle")
    ap.add_argument("--solver", default="cg.mg", help="cg.mg | cg.blockdiagonal | cg.diagonal | cg.identity")
    ap.add_argument("--no-jacobi", action="store_true", help="skip the extra Jacobi-CG solve reported next to --solver")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed "
                                                          "(solution, system matrix values, rhs; a fixed seeded sample of "
                                                          "at most %d entries each) as DIR/<name>.npy" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the GPU path computed; the reference arm has no such outputs")
        if args.cpu_cg_iters <= 0:
            n_cpu = args.cpu_n if args.cpu_n > 0 else default_cpu_n(args.n)
            args.cpu_cg_iters = max(3, int(100 * (768.0 / n_cpu) ** 2))
        return run_reference(args)
    if args.cpu_n <= 0:
        args.cpu_n = 768
    if args.cpu_cg_iters <= 0:
        args.cpu_cg_iters = max(3, int(100 * (768.0 / args.cpu_n) ** 2))

    import torch
    import dune_hdd_b200 as hdd
    from dune_hdd_b200 import capi
    import ctypes as C

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    comm = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        comm = hdd.parallel.init_comm(rank, world, local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    n = args.n
    parts = (8, 8) if n % 8 == 0 else (1, 1)
    t0 = time.perf_counter()
    grid = hdd.grids.cube(n, partitions=parts, pinned=True)  # page-locked host arrays (hdd_host_alloc)
    t_grid = time.perf_counter() - t0
    problem = hdd.problems.ESV2007()
    roff = hdd.parallel.rank_cell_offsets(grid, world)
    cell_range = (int(roff[rank]), int(roff[rank + 1]))
    options = {"type": args.solver, "precision": PRECISION, "max_iter": 200000}

    def make():
        d = hdd.BlockSWIPDG(grid, problem, device=local_rank, cell_range=cell_range, comm=comm)
        return d

    d = make()
    d.init()
    n_dofs = d.num_dofs()
    launches0 = capi.kernel_launches()

    def step():
        ta = d.assemble()
        _, info = d.uncached_solve(options, return_info=True, copy_to_host=False)
        return ta, info

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    launches1 = capi.kernel_launches()
    t0 = time.perf_counter()
    results = [step() for _ in range(args.steps)]
    barrier()
    wall = time.perf_counter() - t0
    launches = capi.kernel_launches() - launches1
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d, torch, capi, rank, world)

    t_asm = sum(r[0] for r in results)
    t_cg = sum(r[1]["seconds"] for r in results)
    iters = results[-1][1]["iterations"]
    stats = torch.tensor([t_asm, t_cg, wall] + [r[0] + r[1]["seconds"] for r in results], dtype=torch.float64, device="cuda")
    if world > 1:
        torch.distributed.all_reduce(stats, op=torch.distributed.ReduceOp.MAX)
    t_asm, t_cg, wall = [float(v) for v in stats.cpu()[:3]]
    step_ms = [1e3 * float(v) for v in stats.cpu()[3:]]  # per step, max over ranks: shows an outlier step for what it is

    # ---- what was timed is checked: true residual recomputed from scratch, error against the exact solution ----------
    res, floor = d.residual(with_floor=True)
    # b scales with h^2 against O(1) matrix entries: recomputing b - A x in fp64 has a rounding level of its own (`floor`,
    # an upper estimate), below which no solver can push it; the solve itself is judged by the error norms below
    check = {"true_residual": res, "true_residual_fp64_floor": floor, "true_residual_bound": max(1e-9, 0.25 * floor),
             "cg_iterations": iters}
    norms = d.error_norms(*hdd.problems.ESV2007_EXACT, order=5)
    # asymptotics of the committed SGrid ladder (test/linearelliptic-swipdg-expectations_esv2007_2dsgrid.cxx:32-36):
    # L2 n^2 = 0.723, 0.742, 0.759, 0.770 -> 0.78; H1 n = 2.216, 2.224, 2.234, 2.240 -> 2.25
    check.update({"L2_error": norms["L2"], "H1_semi_error": norms["H1_semi"], "energy_error": norms["energy"],
                  "H1_semi_expected": 2.25 / n, "L2_expected": 0.78 / (n * n)})
    check_ok = (check["true_residual"] <= check["true_residual_bound"] and
                (n < 64 or (abs(norms["H1_semi"] - 2.25 / n) <= 0.02 * 2.25 / n and
                            abs(norms["L2"] - 0.78 / (n * n)) <= 0.05 * 0.78 / (n * n))))

    # the plain Jacobi-preconditioned CG on the same system, once, outside the timed steps: its SpMV / update / direction
    # kernels are the ones the roofline numbers below are taken from
    jacobi = None
    if not args.no_jacobi or args.solver != "cg.diagonal":
        jopt = dict(options, type="cg.diagonal")
        if args.no_jacobi:
            jopt["max_iter"] = 50
        try:
            _, ji = d.uncached_solve(jopt, return_info=True, copy_to_host=False)
        except hdd.discretizations.linear_solver_failed:
            ji = None
        if ji is not None:
            js = torch.tensor([ji["seconds"]], dtype=torch.float64, device="cuda")
            if world > 1:
                torch.distributed.all_reduce(js, op=torch.distributed.ReduceOp.MAX)
            jacobi = {"solve_s": float(js.cpu()[0]), "iterations": ji["iterations"],
                      "s_per_iteration": float(js.cpu()[0]) / max(ji["iterations"], 1),
                      "halo": ("peer-memory SpMV (CUDA IPC over NVLink)" if ji.get("peer_memory") else "NCCL send/recv")
                      if world > 1 else "none"}

    # roofline of the dominant kernel: CG SpMV, timed alone with CUDA events on the library's stream
    L = capi.lib()
    roof = {}
    peak, peak_kind = measured_peak_gbs()
    # DRAM traffic per launch from the committed `ncu --set full` capture of this workload (profiles/), if it matches
    traffic = {}
    for fname, kmap in (("r01c_traffic_n4096.json", {"cg_update": "k_cg_update", "cg_direction": "k_cg_direction"}),
                        ("r01f_traffic_n4096.json", {"spmv": "k_cg_spmv_tma", "assembly": "k_assemble_lhs_cube<0, 4, 1>"})):
        try:
            with open(os.path.join(ROOT, "profiles", fname)) as f:
                tj = json.load(f)
            if tj.get("cells") == n * n and world == 1:
                traffic.update({k: tj["kernels"][v]["dram_bytes"] for k, v in kmap.items() if v in tj["kernels"]})
        except Exception:
            pass
    for which, name in ((0, "spmv"), (1, "cg_update"), (2, "cg_direction"), (3, "assembly")):
        sec, byt = C.c_double(), C.c_double()
        capi.check(L.hdd_profile_kernel(d._h, which, 20 if which != 3 else 5, C.byref(sec)))
        capi.check(L.hdd_kernel_bytes(d._h, which, C.byref(byt)))
        roof[name] = {"bound": "hbm", "achieved": byt.value / sec.value / 1e9, "peak": peak, "unit": "GB/s",
                      "frac": byt.value / sec.value / 1e9 / peak, "traffic": traffic.get(name), "ms": sec.value * 1e3,
                      "algorithmic_bytes": byt.value, "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)"}

    # the same solver on the CPU baseline's solve sample (cg.diagonal on cpu_solve_n^2 cells): a same-size pair for the
    # "CG solve s" half of the metric
    same_size = None
    if world == 1 and not args.no_cpu_baseline:
        gs = hdd.grids.cube(args.cpu_solve_n)
        ds = hdd.SWIPDG(gs, problem, device=local_rank)
        ds.init()
        _, si = ds.uncached_solve(dict(options, type="cg.diagonal"), return_info=True, copy_to_host=False)
        _, sm = ds.uncached_solve(dict(options, type="cg.mg"), return_info=True, copy_to_host=False)
        same_size = {"grid": "%dx%d" % (args.cpu_solve_n, args.cpu_solve_n), "cg.diagonal_s": si["seconds"],
                     "cg.diagonal_iterations": si["iterations"], "cg.mg_s": sm["seconds"], "cg.mg_iterations": sm["iterations"]}
        del ds

    # end to end through the public API from host buffers (H2D of the grid + problem, D2H of the solution), every step
    e2e = None
    del d
    torch.cuda.empty_cache()
    if not args.no_e2e:
        e_asm, e_cg = [], []
        own_dofs = (cell_range[1] - cell_range[0]) * 4
        x_host = capi.pinned_empty((own_dofs,), np.float64)  # page-locked result buffer, reused by every step
        e2e_warm = max(1, min(args.warmup, 3))  # untimed end-to-end steps first (allocator, peer mappings of new blocks)
        for k in range(e2e_warm + args.steps):
            barrier()
            if k == e2e_warm:
                h2d0 = capi.h2d_bytes()
            t0 = time.perf_counter()
            d2 = make()
            d2.init()
            d2._sync = capi.check(L.hdd_sync(d2._h))
            t1 = time.perf_counter()
            u, info = d2.uncached_solve(options, return_info=True, copy_to_host=True, out=x_host)
            t2 = time.perf_counter()
            del d2
            if k >= e2e_warm:
                e_asm.append(t1 - t0)
                e_cg.append(t2 - t1)
        ev = torch.tensor([sum(e_asm), sum(e_cg)], dtype=torch.float64, device="cuda")
        if world > 1:
            torch.distributed.all_reduce(ev, op=torch.distributed.ReduceOp.MAX)
        ea, ec = [float(v) for v in ev.cpu()]
        own_cells = cell_range[1] - cell_range[0]
        # bytes the library copied host -> device during the timed steps (counted at every copy), summed over the ranks
        hb = torch.tensor([float(capi.h2d_bytes() - h2d0) / args.steps], dtype=torch.float64, device="cuda")
        if world > 1:
            torch.distributed.all_reduce(hb)
        h2d = float(hb.cpu()[0])
        e2e = {"value": args.steps * n_dofs / ea, "unit": "DoFs/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(n_dofs * 8), "cg_solve_s": ec / args.steps,
               "setup_s": ea / args.steps, "setup_steps_s": [round(v, 5) for v in e_asm],
               "note": "value = DoFs / (hdd_mesh_create from page-locked host arrays + hdd_swipdg_create + init), incl. "
                       "host-side localisation of the grid; cg_solve_s includes the D2H copy of the solution; the expanded CSR "
                       "index arrays (a consumer view no kernel reads, 3.1 ms to write) are built at the first hdd_pattern call"}

    # the same end to end with the grid provider's three vectors instead of flat arrays (hdd_mesh_create_cube: what the
    # reference's own test case hands over, testcases/ESV2007.hh:123-127); reported next to `e2e`, which keeps the host arrays
    if e2e is not None:
        provider = hdd.grids.CubeProvider(n, partitions=parts)
        p_asm, p_cg = [], []
        for k in range(e2e_warm + args.steps):
            barrier()
            if k == e2e_warm:
                h2d0 = capi.h2d_bytes()
            t0 = time.perf_counter()
            d2 = hdd.BlockSWIPDG(provider, problem, device=local_rank, cell_range=cell_range, comm=comm)
            d2.init()
            capi.check(L.hdd_sync(d2._h))
            t1 = time.perf_counter()
            u, info = d2.uncached_solve(options, return_info=True, copy_to_host=True, out=x_host)
            t2 = time.perf_counter()
            del d2
            if k >= e2e_warm:
                p_asm.append(t1 - t0)
                p_cg.append(t2 - t1)
        pv = torch.tensor([sum(p_asm), sum(p_cg)], dtype=torch.float64, device="cuda")
        if world > 1:
            torch.distributed.all_reduce(pv, op=torch.distributed.ReduceOp.MAX)
        pa, pc = [float(v) for v in pv.cpu()]
        hb = torch.tensor([float(capi.h2d_bytes() - h2d0) / args.steps], dtype=torch.float64, device="cuda")
        if world > 1:
            torch.distributed.all_reduce(hb)
        p_h2d = float(hb.cpu()[0])
        e2e["cube_provider"] = {"value": args.steps * n_dofs / pa, "unit": "DoFs/s", "setup_s": pa / args.steps,
                                "cg_solve_s": pc / args.steps, "h2d_bytes_per_step": int(p_h2d),
                                "d2h_bytes_per_step": int(n_dofs * 8),
                                "note": "hdd_mesh_create_cube(lower_left, upper_right, num_elements, partition): grid tables "
                                        "written on the device"}

    est, est_ok = (None, True)
    if not args.no_estimator:
        est, est_ok = estimator_phase(hdd, torch, capi, comm, rank, world, local_rank, n, peak, peak_kind, barrier)
    parity, parity_ok = (None, True)
    if not args.no_parity:
        parity, parity_ok = small_grid_parity(hdd, torch, comm, rank, world, local_rank)
    check["small_grid_parity"] = parity
    check["ok"] = bool(check_ok and est_ok and parity_ok)

    if rank == 0:
        config = workload_config(n, args.solver, world)
        config["halo"] = (("peer-memory SpMV (CUDA IPC over NVLink)" if results[-1][1].get("peer_memory") else
                           "NCCL send/recv of the CG direction" + (", row-strip exchanges of the vertex levels (cg.mg)"
                                                                  if args.solver == "cg.mg" else ""))
                          if world > 1 else "none")
        line = {"metric": METRIC, "value": args.steps * n_dofs / t_asm, "unit": "DoFs/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "step_ms": step_ms,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config,
                "assemble_ms": 1e3 * t_asm / args.steps, "cg_solve_s": t_cg / args.steps, "cg_iterations": iters,
                "cg_s_per_iteration": t_cg / args.steps / max(iters, 1), "cg_diagonal": jacobi,
                "time_to_solution_dofs_per_s": n_dofs / (wall / args.steps),
                "check": check,
                "roofline": roof["spmv"], "roofline_assembly": roof["assembly"], "roofline_cg_update": roof["cg_update"],
                "roofline_cg_direction": roof["cg_direction"], "estimator": est, "same_size_solve": same_size,
                "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "grid_generation_s": t_grid}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.cpu_n, args.cpu_cg_iters, args.cpu_solve_n)
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()
    if not check["ok"]:
        sys.stderr.write("bench.py: the in-run check failed: %s\n" % json.dumps(check))
        sys.exit(3)


if __name__ == "__main__":
    main()
