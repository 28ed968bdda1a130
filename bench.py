#!/usr/bin/env python
"""bench.py — one Newton step of the hot path (assemble_system + solve_system) on a synthetic
uniformly refined cylinder mesh, N GPUs of one node (one process per GPU).

  python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
  python bench.py --dump-outputs bench_outputs ...          # + what the last timed step computed, as .npy (see dump_outputs)
  python bench.py --impl reference ...                      # the CPU oracle port on the host cores
  python bench.py --precond block_diagonal                  # opt-in: the CONVERGED preconditioned solve of BASELINE.json configs[1]
                                                            # (one GPU, ~80 s, its own JSON line; see run_precond)

A "step" = zero-free owner-computes assembly of J, Mp, R (+ Neumann) + Dirichlet rows + ||R|| +
GMRES(28, identity) capped at --gmres-its steps (the synthetic state does not converge with an
unpreconditioned GMRES, exactly like the CPU oracle; the cap makes the step deterministic).
metric = BASELINE.json's "Jacobian assembly MDoF/s" (value) with "GMRES time per Newton step"
reported beside it in the same JSON line.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MESHES = {  # name -> (file, surface entity, geometric tags?, Dirichlet calls, neumann id, inlet)
    "cmy": ("cylinder_cmy.msh", -1, False, [{11: True}, {11: True, 12: False, 13: False}], 10,
            dict(u_m=1.5, H=0.41, y0=0.0)),
    "mesh2d": ("cylinder_mesh2d.msh", 5, True, [{0: True}, {2: False, 3: False}], 1, dict(u_m=1.5, H=4.1, y0=-2.0)),
}


def analytic_state(xy, n_u):
    """Synthetic iterate u = (sin(pi x) cos(pi y), -cos(pi x) sin(pi y)), p = x y at the support points (85 M of them at the default
    size: evaluated with torch's multi-threaded CPU kernels when torch is there, numpy otherwise)."""
    sol = np.zeros(len(xy))
    torch = sys.modules.get("torch")  # only if the caller has it loaded already (the CPU-baseline workers do not)
    if torch is not None:
        t, out = torch.from_numpy(xy), torch.from_numpy(sol)
        x0, y0, x1, y1 = t[0:n_u:2, 0], t[0:n_u:2, 1], t[1:n_u:2, 0], t[1:n_u:2, 1]
        out[0:n_u:2] = torch.sin(np.pi * x0) * torch.cos(np.pi * y0)
        out[1:n_u:2] = -torch.cos(np.pi * x1) * torch.sin(np.pi * y1)
        out[n_u:] = t[n_u:, 0] * t[n_u:, 1]
    else:
        sol[0:n_u:2] = np.sin(np.pi * xy[0:n_u:2, 0]) * np.cos(np.pi * xy[0:n_u:2, 1])
        sol[1:n_u:2] = -np.cos(np.pi * xy[1:n_u:2, 0]) * np.sin(np.pi * xy[1:n_u:2, 1])
        sol[n_u:] = xy[n_u:, 0] * xy[n_u:, 1]
    return sol


def build_problem(pkg, mesh, levels, world, rank, patterns=True):
    fn, ent, geo, calls, neumann, inlet = MESHES[mesh]
    m = pkg.Mesh.read_msh(os.path.join(ROOT, "tests", "golden", fn), ent)
    if geo:
        m.tag_boundary_box(0, 1, 2, 3)
    if levels:
        m = m.refine(levels)
    cp = m.partition_rcb(world) if world > 1 else None
    d = pkg.Dofs(m, world, cp)
    part = pkg.Part(d, rank, patterns=patterns)   # patterns=False: built on the device (SURVEY 8f N4)
    gd, gv = d.dirichlet_values(calls, dict(time_factor=1.0, **inlet))
    ld, lv = part.localize_dirichlet(gd, gv)
    xy = d.support_points()
    sol = analytic_state(xy, d.n_u)[part.l2g[: part.n_own]]
    return m, d, part, (ld, lv), neumann, sol


class ClockSampler:
    """SM clock / throttle reasons of one GPU DURING the timed region (B200_PROFILING.md's clocks line). Polls NVML in-process every
    10 ms (the timed region of the 8-GPU run lasts half a second: an `nvidia-smi -lms` child does not deliver its first row in that
    time on an 8-GPU host); falls back to the nvidia-smi loop when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASONS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc, self.nvml, self.stop_flag = gpu, [], None, None, threading.Event()
        self.sm, self.mask, self.sm_max, self.source = [], 0, None, None

    def start(self):
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(self.gpu)
            bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
            self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml, self.source = pynvml, "nvml, 10 ms"
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:  # noqa: BLE001  (no NVML: try the command-line tool)
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.source = "nvidia-smi -lms 100"
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                self.mask |= int(reasons(self.handle))
            except Exception:  # noqa: BLE001
                pass
            self.stop_flag.wait(0.010)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([s.strip() for s in line.split(",")])

    def stop(self):
        if self.nvml:
            self.stop_flag.set()
            self.thread.join(timeout=1.0)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max, "samples": len(self.sm),
                    "reasons": sorted(n for n, bit in self.REASONS if self.mask & bit), "source": self.source}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(self.rows[0][2]) if self.rows and len(self.rows[0]) >= 9 else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": self.source}


def _cpulist(txt):
    cpus = set()
    for part in txt.strip().split(","):
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa_node(local_rank):
    """Pin this process (and the pinned host buffers it first-touches afterwards) to the CPUs next to its GPU: with 8 ranks on a
    two-socket host the H2D copies of the e2e step otherwise cross the socket link. Sources, in order: sysfs numa_node of the GPU's
    PCI device, the "CPU Affinity" column of `nvidia-smi topo -m`. Returns a short description for the JSON line; a no-op when
    neither tells."""
    import re
    try:
        import torch
        prop = torch.cuda.get_device_properties(local_rank)
        path = f"/sys/bus/pci/devices/{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node >= 0:
            allowed = _cpulist(open(f"/sys/devices/system/node/node{node}/cpulist").read()) & os.sched_getaffinity(0)
            if allowed:
                os.sched_setaffinity(0, allowed)
                return f"numa node {node} (sysfs), {len(allowed)} cpus"
    except Exception:  # noqa: BLE001
        pass
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        for line in out.splitlines():
            cols = re.split(r"\s{2,}|\t", re.sub(r"\x1b\[[0-9;]*m", "", line.strip()))
            if not cols or cols[0] != f"GPU{local_rank}":
                continue
            for tok in cols[1:]:
                if re.fullmatch(r"\d+(-\d+)?(,\d+(-\d+)?)*", tok) and ("-" in tok or "," in tok):
                    allowed = _cpulist(tok) & os.sched_getaffinity(0)
                    if allowed:
                        os.sched_setaffinity(0, allowed)
                        return f"cpu affinity {tok} (nvidia-smi topo), {len(allowed)} cpus"
        return "not bound (no affinity information)"
    except Exception as e:  # noqa: BLE001
        return f"not bound ({type(e).__name__})"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_baseline_assembly(pkg, mesh, level, workers, start="fork"):
    """Oracle (CPU port of the reference loops) assembling `workers` independent replicas of the
    level-`level` mesh, one per process: the perfect-scaling upper bound of `mpirun -np workers`."""
    if workers == 1:
        r = _oracle_worker((mesh, level))
        return r[0], r[1], r[2], r[3]
    import multiprocessing as mp
    ctx = mp.get_context(start)   # "spawn" from a process that holds a CUDA context (the GPU arm)
    with ctx.Pool(workers) as pool:
        res = pool.map(_oracle_worker, [(mesh, level)] * workers)
    n = res[0][0]
    t_asm = max(r[1] for r in res)
    t_it = max(r[2] for r in res)
    return n, t_asm, t_it, res[0][3]


def _oracle_worker(args):
    mesh, level = args
    pkg = importlib.import_module("navier-stokes-dealii_b200")
    from oracle.oracle import Oracle
    m, d, part, (ld, lv), neumann, sol = build_problem(pkg, mesh, level, 1, 0)
    o = Oracle(part)
    o.set_params(neumann_id=neumann)
    o.set_solution(sol)
    o.set_solution_old(0.9 * sol)
    t0 = time.perf_counter()
    o.assemble()
    o.apply_dirichlet(ld, lv)
    t_asm = time.perf_counter() - t0
    t0 = time.perf_counter()
    its, res, rc = o.solve(0, 1e-2, 28, 30, 0)
    t_solve = time.perf_counter() - t0
    return d.n, t_asm, t_solve / max(its, 1), m.n_cells


def run_reference(args):
    """--impl reference: the reference's CPU path = the oracle port (deal.II/Trilinos/MPI are not in
    this image, SURVEY §8c), all host cores, bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["OMP_NUM_THREADS"] = "1"   # one core per replica
    pkg = importlib.import_module("navier-stokes-dealii_b200")
    workers = os.cpu_count() or 1
    level = args.cpu_level
    vals, its = [], []
    for s in range(args.warmup + args.steps):
        n, t_asm, t_it, cells = cpu_baseline_assembly(pkg, args.mesh, level, workers)
        if s >= args.warmup:
            vals.append(workers * n / t_asm / 1e6)
            its.append(t_it / workers)
    v = float(np.mean(vals))
    sample = (f"{workers} independent replicas (one per core, perfect-scaling bound of mpirun -np {workers}) of the "
              f"{args.mesh} mesh refined {level}x ({cells} cells, {n} DoFs each); assembly + Dirichlet timed")
    line = {"impl": "reference", "metric": "jacobian_assembly_mdofs", "value": v, "unit": "MDoF/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(1e3 * n * workers / (v * 1e6)),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(workload_config(args, None), levels=level, full_workload_levels=args.levels, cells=int(cells),
                           dofs=int(n), sample=sample),
            "gmres_ms_per_iteration_per_replica_dof": None,
            "cpu_baseline": {"value": v, "unit": "MDoF/s", "cores": workers, "kind": "port", "sample": sample,
                             "gmres_s_per_iteration_at_sample_size": float(np.mean(its)) * workers},
            "e2e": {"value": v, "unit": "MDoF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


DUMP_SAMPLE = 1 << 20   # global DoFs drawn for the dumped vectors: ~25 MB in all at the default size (85 M DoFs)
DUMP_ROWS = 1 << 14     # global rows drawn for the dumped matrix entries: ~0.5 M entries of J, ~13 MB, at the default size


def _sample(n, k, seed):
    """All of range(n) up to k ids, else the sorted unique ids of k draws of a generator seeded with `seed`."""
    return np.arange(n) if n <= k else np.unique(np.random.default_rng(seed).integers(0, n, k))


def _rows_entries(rp, col, rows, l2g):
    """Global (row, column) and CSR position of every stored entry of the local CSR rows `rows`."""
    lens = rp[rows + 1] - rp[rows]
    pos = np.repeat(rp[rows], lens) + np.arange(lens.sum()) - np.repeat(np.cumsum(lens) - lens, lens)
    return np.repeat(l2g[rows], lens), l2g[col[pos]], pos


def dump_outputs(out_dir, d, part, dev, r, its, res, rank, world, dist):
    """--dump-outputs: write what the last timed step computed to out_dir as float64 .npy files, so that two builds can be
    compared output for output.  Every rank takes part; rank 0 writes.
      sample_dofs                      global DoF ids of the vector sample: _sample(n, DUMP_SAMPLE, seed 0)
      newton_increment                 the GMRES increment (get_delta) at sample_dofs
      residual                         the right-hand side after the Dirichlet rows (get_residual) at sample_dofs
      jacobian_{rows,cols,values}      every stored entry of J (after the Dirichlet rows) in the global rows
                                       _sample(n, DUMP_ROWS, seed 1), keyed by global (row, column), in that order
      pressure_mass_{rows,cols,values} the same for the pressure mass matrix Mp (its velocity rows are empty)
      gmres_residual_history           the residual norm after every GMRES step
      step_scalars                     [||R||, GMRES steps, final GMRES residual]
    The sample depends on n alone: the same ids for the same arguments."""
    n = int(d.n)
    dofs, rows = _sample(n, DUMP_SAMPLE, 0), _sample(n, DUMP_ROWS, 1)
    own = part.l2g[: part.n_own]
    picked = np.zeros(n, bool)
    picked[dofs] = True
    sel = np.flatnonzero(picked[own])
    picked[:] = False
    picked[rows] = True
    rsel = np.flatnonzero(picked[own])
    out = {"vectors": (own[sel], dev.get_delta()[sel], dev.get_residual()[sel])}
    rp, col, prp, pcol = dev.get_pattern()
    jac, pm = _rows_entries(rp, col, rsel, part.l2g), _rows_entries(prp, pcol, rsel, part.l2g)
    del rp, col, prp, pcol          # the whole pattern and then all nnz(J) values pass through the host, one after the other
    out["jacobian"] = jac[:2] + (dev.get_matrix_values()[jac[2]],)
    out["pressure_mass"] = pm[:2] + (dev.get_pm_values()[pm[2]],)
    history = dev.gmres_history()
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, out)
        out = {k: tuple(np.concatenate(a) for a in zip(*(g[k] for g in gathered))) for k in out}
    if rank != 0:
        return
    g, delta, rhs = out["vectors"]
    order = np.argsort(g)
    assert np.array_equal(g[order], dofs)
    files = {"sample_dofs": dofs, "newton_increment": delta[order], "residual": rhs[order],
             "gmres_residual_history": history, "step_scalars": [r, its, res]}
    for name in ("jacobian", "pressure_mass"):
        i, j, v = out[name]
        order = np.lexsort((j, i))
        files.update({f"{name}_rows": i[order], f"{name}_cols": j[order], f"{name}_values": v[order]})
    os.makedirs(out_dir, exist_ok=True)
    for name, a in files.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, np.float64))


def workload_config(args, d):
    cfg = {"workload": f"synthetic uniformly refined cylinder mesh: {MESHES[args.mesh][0]} red-refined {args.levels}x, "
                       "P2-P1, state u=(sin(pi x)cos(pi y), -cos(pi x)sin(pi y)), p=xy, u_old=0.9u",
           "mesh": args.mesh, "levels": args.levels, "gmres_its_cap": args.gmres_its, "nu": args.nu, "deltat": args.deltat,
           "preconditioner": "identity (reference cpp:570)", "l2": "inputs larger than L2 (no flush needed)",
           "parallelism": f"mesh partition x{args.gpus} (RCB), ghost-layer owner-computes assembly, halo exchange by NVLink peer stores, Krylov all-reduce fused "
                          "into the reduction kernels (NVLink peer memory)"}
    if d is not None:
        cfg.update({"cells": int(d.mesh.n_cells), "dofs": int(d.n)})
    return cfg


def run_precond(args):
    """--precond: BASELINE.json configs[1] at its stated size - mesh-square-h0.012500.msh (12 800 cells, 58 403 DoFs), Stokes-initialised
    steady Navier-Stokes through the reference's block preconditioners (hpp:520-639), the largest repo mesh on which the reference's
    own inner-solver settings converge (profiles/r02_summary.md section 6).  One GPU.  Prints ONE JSON line of its own: the converged
    "GMRES time per Newton step" VERDICT r1 asked for beside the capped identity figure of the default run, with the ILU(0) apply
    (the kernel that bounds it) timed on the device for every triangular-solve variant and put against the HBM roofline."""
    import importlib
    import torch
    pkg = importlib.import_module("navier-stokes-dealii_b200")
    torch.cuda.set_device(0)
    prm = pkg.Parameters(mesh_path=os.path.join(ROOT, "tests", "golden", "square_h0.0125.msh"), nu=0.05, H=1.0, inlet_time_mode="constant",
                         neumann_id=1, inlet_id=0, wall_ids=(2, 3), clear_inlet_before_walls=True, use_mass=False,
                         preconditioner=args.precond, p_out=0.0, increment_bc="consistent", newton_max_iters=8)
    mesh = pkg.Mesh.read_msh(prm.mesh_path, prm.surface_entity)
    s = pkg.NavierStokesSolver(2, 1, 1.0, 1.0, prm, verbose=False)
    t0 = time.perf_counter()
    s.setup(mesh)
    setup_s = time.perf_counter() - t0
    dev = s.dev
    solves = []
    plain_solve = dev.solve

    def timed_solve(*a, **k):
        t = time.perf_counter()
        out = plain_solve(*a, **k)
        solves.append({"outer_gmres_steps": int(out[0]), "inner_iterations": dev.last_inner_iterations(),
                       "device_ms": dev.phase_ms()["solve"], "wall_ms": 1e3 * (time.perf_counter() - t)})
        return out
    dev.solve = timed_solve
    sampler = ClockSampler(0)
    sampler.start()
    t0 = time.perf_counter()
    error = None
    try:
        s.solve(stokes_init=True)
    except Exception as e:  # noqa: BLE001  (e.g. the inner CG of the block-triangular preconditioner does not converge on this system)
        error = f"{type(e).__name__}: {e}"
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    hbm, hbm_src = peaks()
    d = s.dofs
    rp, cl = dev.get_pattern()[:2]
    n_u, n_p = int(d.n_u), int(d.n_p)
    nnz_A = int((cl[: rp[n_u]] < n_u).sum())
    ilu = {}
    for variant, label in ((0, "one launch per level"), (1, "stamped single launch, all SMs"), (2, "one CTA, shared-memory window"),
                           (-1, "library's choice")):
        dev.set_tuning(4, variant)
        dev.time_kernel(6, 2)
        ilu[label] = {"A_ms": dev.time_kernel(6, 20), "Mp_ms": dev.time_kernel(7, 20)}
    dev.set_tuning(4, -1)
    a_ms = ilu["library's choice"]["A_ms"]
    a_bytes = 12 * nnz_A + 24 * n_u   # factors + column indices once, right-hand side, unknowns
    inner = sum(x["inner_iterations"] for x in solves)
    line = {"metric": "preconditioned_newton_solve_s", "value": wall, "unit": "s", "n_gpus": 1, "higher_is_better": False, "dtype": "f64",
            "data": "the reference's own mesh", "impl": "b200",
            "error": error,
            "config": {"workload": "BASELINE.json configs[1]: mesh-square-h0.012500.msh, Stokes-initialised steady Navier-Stokes, nu = 0.05, "
                                   "reference tolerances (outer GMRES 1e-2, inner 1e-2, cpp:566, hpp:541-612)",
                       "preconditioner": args.precond, "cells": int(mesh.n_cells), "dofs": int(d.n)},
            "newton_history": [[int(a), int(b), float(c), None if e is None else int(e)] for a, b, c, e in s.history],
            "solves": solves, "gmres_ms_per_newton_step": float(np.mean([x["device_ms"] for x in solves])) if solves else None,
            "inner_iterations_total": inner, "ilu_applies_share_of_solve_time_upper_bound":
                (inner * a_ms) / max(sum(x["device_ms"] for x in solves), 1e-9),
            "ilu_apply_device_ms": ilu, "setup_s": setup_s, "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_ilu_solve_cta<lower> + <upper> (ILU(0) apply of the velocity block)",
                         "achieved": a_bytes / a_ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": a_bytes / a_ms / 1e6 / hbm, "traffic": None,
                         "peak_source": hbm_src, "algorithmic_bytes_per_launch": a_bytes, "ms_per_launch": a_ms,
                         "note": "a dependency chain of 1 120 + 1 120 levels of ~46 rows: bound by the latency of a level (0.76 us), not by "
                                 "bytes - the HBM fraction is reported for completeness"}}
    print(json.dumps(line), flush=True)
    dev.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    # default workload = BASELINE.json configs[3]: the cylinder domain (surface entity 5 of mesh2d.msh) red-refined
    # 8x = 18.9 M triangles, 85 M DoFs ("~16M triangles, ~70M DoFs"); --mesh cmy --levels 5 is the 6.6 M-cell case
    ap.add_argument("--mesh", default="mesh2d", choices=list(MESHES))
    ap.add_argument("--levels", type=int, default=8)
    ap.add_argument("--gmres-its", type=int, default=56)
    ap.add_argument("--cpu-level", type=int, default=None, help="refinement level of the CPU-baseline sample")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="weak (BASELINE.json configs[4]): --levels is the 1-GPU level, N GPUs refine floor(log4 N) more")
    ap.add_argument("--viscosity", dest="nu", type=float, default=0.001, help="viscosity (reference hpp:703; configs[4]: 5e-4 = Re 200)")
    ap.add_argument("--time-step", dest="deltat", type=float, default=0.05, help="time step (reference main.cpp:13; configs[4]: small)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--host-patterns", action="store_true", help="build the sparsity patterns on the host (libnst) and upload them")
    ap.add_argument("--precond", default=None, choices=["block_triangular", "block_diagonal"],
                    help="instead of the default run: the converged preconditioned solve of BASELINE.json configs[1] (one GPU, own JSON line)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.precond or args.impl != "b200"):
        ap.error("--dump-outputs applies to the default run of the CUDA path")
    if args.precond:
        return run_precond(args)
    if args.cpu_level is None:
        args.cpu_level = {"cmy": 2, "mesh2d": 4}[args.mesh]
    if args.scaling == "weak":      # cells per GPU: 1x, 1/2x, 1x, 1/2x of the 1-GPU mesh at N = 1, 2, 4, 8
        args.base_levels = args.levels
        args.levels = args.levels + int(np.floor(np.log(max(args.gpus, 1)) / np.log(4) + 1e-9))
    # torchrun exports OMP_NUM_THREADS=1; the host topology code (libnst.so) is OpenMP-parallel
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl != "reference":
        os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // world_env))
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else "single rank: not bound"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("navier-stokes-dealii_b200")

    t_setup = time.perf_counter()
    m, d, part, (ld, lv), neumann, sol = build_problem(pkg, args.mesh, args.levels, world, rank, patterns=args.host_patterns)
    t_topology = time.perf_counter() - t_setup
    dev = pkg.DeviceProblem(part, local)
    if world > 1:
        uid = [pkg.DeviceProblem.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        dev.comm_init(rank, world, uid[0])
        peer_ar = dev.enable_peer_allreduce(dist)
    dev.set_params(neumann_id=neumann, nu=args.nu, deltat=args.deltat)
    dev.set_solution(sol)
    dev.set_solution_old(0.9 * sol)
    t_setup = time.perf_counter() - t_setup
    N = d.n
    zero = np.zeros(part.n_own)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        dev.assemble()
        dev.apply_dirichlet(ld, lv)
        r = dev.residual_norm()
        its, res, rc = dev.solve(0, 1e-2, args.gmres_its, 30, 0, check=False)
        if rc not in (0, -3):
            raise RuntimeError(f"nsg_solve failed: {rc}")
        ph = dev.phase_ms()
        return r, its, res, ph

    e2e_parts = []

    def step_e2e(host_sol):
        t0 = time.perf_counter()
        dev.set_solution(host_sol)                 # H2D from pinned host memory: the step's input iterate
        t1 = time.perf_counter()
        dev.assemble()
        t2 = time.perf_counter()
        dev.apply_dirichlet(ld, lv)
        t3 = time.perf_counter()
        r = dev.residual_norm()                    # D2H: the step's result (assembly metric)
        t_asm = time.perf_counter() - t0
        e2e_parts.append((t1 - t0, t2 - t1, t3 - t2, t0 + t_asm - t3))
        its, res, rc = dev.solve(0, 1e-2, args.gmres_its, 30, 0, check=False)
        delta = dev.get_delta(host_delta)          # D2H into pinned host memory: the Newton increment
        return t_asm, time.perf_counter() - t0, delta

    for _ in range(args.warmup):
        dev.set_delta(zero)
        step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    c0 = dev.counters()
    asm_ms, dir_ms, sol_ms, its_seen = [], [], [], []
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        dev.set_delta(zero)
        r, its, res, ph = step()
        asm_ms.append(ph["assemble"]), dir_ms.append(ph["dirichlet"]), sol_ms.append(ph["solve"])
        its_seen.append(its)
    ev1.record()
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    c1 = dev.counters()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:      # before the kernel timings and the extra solves below overwrite the device state
        dump_outputs(args.dump_outputs, d, part, dev, r, its, res, rank, world, dist)

    # device-timed phases: max over ranks
    local_t = torch.tensor([np.mean(asm_ms) + np.mean(dir_ms), np.mean(sol_ms), wall_ms / args.steps],
                           dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(local_t, op=dist.ReduceOp.MAX)
    t_asm_ms, t_sol_ms, t_step_ms = (float(x) for x in local_t.cpu())
    value = N / (t_asm_ms * 1e-3) / 1e6

    # roofline of the dominant kernel (SpMV: G launches per step) + the other two hot kernels
    hbm, hbm_src = peaks()
    reps = 10
    n_rows, nnz, n_cols = part.n_own, dev.nnz, part.n_loc
    spmv_ms = dev.time_kernel(1, reps)
    spmv_bytes = 12 * nnz + 8 * n_cols + 8 * n_rows + 8 * (n_rows + 1)
    aad_ms = dev.time_kernel(2, reps)
    g_its = int(its_seen[-1])
    mgs_passes = sum(min(i % 28, 27) + 1 for i in range(g_its))   # add_and_dot launches of the MGS sweeps
    asm_k_ms = dev.time_kernel(0, reps)
    fp64_tf = torch.cuda.get_device_properties(local).multi_processor_count * 67108864 * 2 / dev.time_kernel(5, 3) / 1e9
    asm_bytes = (8 * nnz + 8 * dev.pm_nnz + 8 * n_rows + part.n_cells * (15 * 4 + 5 * 8) + 2 * 8 * n_cols)
    traffic = None   # dram__bytes_read+write per launch of the same kernel on the same workload, from profiles/
    tpath = os.path.join(ROOT, "profiles", "spmv_traffic.json")
    if os.path.exists(tpath):
        for rec in json.load(open(tpath)):
            if rec["mesh"] == args.mesh and rec["levels"] == args.levels and rec["n_gpus"] == world:
                traffic = rec["dram_bytes_per_launch"]
    rl = {"bound": "hbm", "kernel": "k_spmv_rowpair<persistent> (SpMV variant 7: CSR, 8 lanes per velocity-node row PAIR sharing one column "
                                   "index and one x gather, prefetched row extents)",
          "achieved": spmv_bytes / spmv_ms / 1e6, "peak": hbm, "unit": "GB/s",
          "frac": spmv_bytes / spmv_ms / 1e6 / hbm, "traffic": traffic, "peak_source": hbm_src,
          "algorithmic_bytes_per_launch": spmv_bytes, "ms_per_launch": spmv_ms,
          "launches_per_step": int(its_seen[-1]) + 2,
          "share_of_step": (int(its_seen[-1]) + 2) * spmv_ms / t_step_ms}
    rl_other = {
        "k_add_and_dot": {"bound": "hbm", "achieved": 32 * n_rows / aad_ms / 1e6, "peak": hbm, "unit": "GB/s",
                          "frac": 32 * n_rows / aad_ms / 1e6 / hbm, "ms_per_launch": aad_ms,
                          "launches_per_step": int(mgs_passes), "share_of_step": mgs_passes * aad_ms / t_step_ms,
                          "note": "modified Gram-Schmidt chain: the largest share of a step; 32 B/DoF per pass"},
        "assembly(k_cell_packets6+k_assemble_u6+k_assemble_p6+k_neumann)": {
            "bound": "hbm", "achieved": asm_bytes / asm_k_ms / 1e6, "peak": hbm, "unit": "GB/s",
            "frac": asm_bytes / asm_k_ms / 1e6 / hbm, "ms_per_launch": asm_k_ms, "algorithmic_bytes_per_launch": asm_bytes,
            "mdofs": part.n_own / asm_k_ms / 1e3,
            "fp64_peak_tflops_measured": fp64_tf,
            "note": "variant 5 (fan scheme); ncu summary and the FP64-pipe share: profiles/r02_summary.md"}}

    # the same GMRES steps with classical Gram-Schmidt (tuning key 3; NOT the reference default): reported beside
    dev.set_tuning(3, 1)
    dev.set_delta(zero)
    dev.solve(0, 1e-2, args.gmres_its, 30, 0, check=False)
    dev.set_delta(zero)
    dev.solve(0, 1e-2, args.gmres_its, 30, 0, check=False)
    cgs_t = torch.tensor([dev.phase_ms()["solve"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(cgs_t, op=dist.ReduceOp.MAX)
    cgs_ms = float(cgs_t.cpu()[0])
    dev.set_tuning(3, 0)

    # end-to-end through the public API with host buffers
    e2e_asm, e2e_step = [], []
    pin_in = torch.empty(part.n_own, dtype=torch.float64).pin_memory()
    pin_out = torch.empty(max(part.n_own, 1), dtype=torch.float64).pin_memory()
    host_sol, host_delta = pin_in.numpy(), pin_out.numpy()
    host_sol[:] = sol
    for _ in range(2):
        step_e2e(host_sol)
    barrier()
    e2e_parts.clear()
    for _ in range(max(2, args.steps // 2)):
        dev.set_delta(zero)
        if world > 1:
            dist.barrier()                         # every rank starts its step together (the halo refresh is a rendezvous)
        a, s, _ = step_e2e(host_sol)
        e2e_asm.append(a), e2e_step.append(s)
    barrier()
    parts_t = torch.tensor(np.mean(np.array(e2e_parts), axis=0), dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(parts_t, op=dist.ReduceOp.MAX)
    e2e_breakdown = [1e3 * float(x) for x in parts_t.cpu()]
    e2e_t = torch.tensor([np.mean(e2e_asm), np.mean(e2e_step)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_asm_s, e2e_step_s = (float(x) for x in e2e_t.cpu())

    if rank == 0:
        line = {"metric": "jacobian_assembly_mdofs", "value": value, "unit": "MDoF/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": t_step_ms, "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args, d),
                "host_binding": numa,
                "assembly_ms": t_asm_ms, "gmres_ms_per_newton_step": t_sol_ms, "gmres_its": int(its_seen[-1]),
                "gmres_ms_per_iteration": t_sol_ms / max(1, its_seen[-1]), "setup_s": t_setup,
                "setup_topology_s": t_topology,
                "gmres_ms_per_newton_step_classical_gs": cgs_ms,
                "krylov_allreduce": ("fused into the reduction kernels (NVLink peer mailboxes)" if world > 1 and peer_ar
                                     else "nccl" if world > 1 else None),
                "gpu_launches": int(c1["launches"] - c0["launches"]), "clocks": clocks, "roofline": rl,
                "roofline_other": rl_other,
                "e2e": {"value": N / e2e_asm_s / 1e6, "unit": "MDoF/s",
                        "h2d_bytes_per_step": int(8 * part.n_own + 12 * len(ld)), "d2h_bytes_per_step": 8,
                        "newton_step_ms": 1e3 * e2e_step_s, "newton_step_d2h_bytes": int(8 + 8 * part.n_own),
                        "breakdown_ms_max_over_ranks": dict(zip(("set_solution_h2d_and_halo", "assemble", "dirichlet",
                                                                 "residual_norm"), e2e_breakdown)),
                        "what": "value: set_solution(host, pinned) + assemble + Dirichlet + residual norm to host (8 bytes back); "
                                "newton_step_ms adds GMRES and get_delta(host), whose bytes are newton_step_d2h_bytes"}}
        if not args.no_cpu_baseline and world == 1:
            # the SAME measurement the reference arm (--impl reference) reports: all host cores, one replica per core
            os.environ["OMP_NUM_THREADS"] = "1"
            workers = os.cpu_count() or 1
            n_s, t_a, t_it, cells = cpu_baseline_assembly(pkg, args.mesh, args.cpu_level, workers, start="spawn")
            line["cpu_baseline"] = {"value": workers * n_s / t_a / 1e6, "unit": "MDoF/s", "cores": workers, "kind": "port",
                                    "sample": f"{workers} independent replicas (one per core, perfect-scaling bound of mpirun -np "
                                              f"{workers}) of the oracle (C++ port of cpp:178-378) on the {args.mesh} mesh refined "
                                              f"{args.cpu_level}x ({cells} cells, {n_s} DoFs each): one assembly + Dirichlet",
                                    "gmres_s_per_iteration_at_sample_size": t_it}
        print(json.dumps(line))
    dev.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
