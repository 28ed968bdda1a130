"""Point evaluation on the default workload (cylinder_mesh2d.msh, surface entity 5, refined 8x: 18.9 M cells, 85 M DoFs):
the spatial index (build time, size, bin occupancy), locate + evaluate of 10^6 random points inside the domain, and the
transfer of a level-7 solution to the support points of level 8 (NavierStokesSolver.set_solution_from).

Kernel times are CUDA events over repeated launches on device-resident points (nsg_time_kernel 8); the full-call times are
host clocks around evaluate() / set_solution_from(), which end in a device synchronise and include the host copies.

Algorithmic bytes per found point: the point (16 B), the chosen cell's grad lambda and first vertex (48 + 16 B), its 15 DoF
indices (60 B) and 15 solution entries (120 B), the values written (24 B) and the global cell id (4 B): 288 B, plus 48 B of
gradients when they are asked for.  The HBM fraction quotes these bytes over the kernel time against 7.7 TB/s (the B200
data-sheet figure); the search through a bin's cells is not counted, so this understates the traffic.

Usage: python scripts/point_eval_time.py [--levels 8] [--points 1000000] [--reps 10]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("navier-stokes-dealii_b200")

HBM_PEAK = 7.7e12
BYTES_VALUES, BYTES_GRADS = 288, 48


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def mesh(levels):
    m = pkg.Mesh.read_msh(os.path.join(ROOT, "tests", "golden", "cylinder_mesh2d.msh"), 5)
    m.tag_boundary_box(0, 1, 2, 3)
    return m.refine(levels) if levels else m


def solver(m):
    s = pkg.NavierStokesSolver(2, 1, 0.05, 0.05, pkg.Parameters(), verbose=False)
    return s.setup(m)


def analytic(s):
    xy = s.dofs.support_points()
    n_u = s.dofs.n_u
    sol = np.empty(s.dofs.n)
    sol[0:n_u:2] = np.sin(np.pi * xy[0:n_u:2, 0]) * np.cos(np.pi * xy[0:n_u:2, 1])
    sol[1:n_u:2] = -np.cos(np.pi * xy[1:n_u:2, 0]) * np.sin(np.pi * xy[1:n_u:2, 1])
    sol[n_u:] = xy[n_u:, 0] * xy[n_u:, 1]
    return sol


def random_points(m, n, seed=0):
    """n points uniform over the domain: cells drawn by area, then uniform barycentric coordinates."""
    xy, cv = m.xy, m.cells
    e1, e2 = xy[cv[:, 1]] - xy[cv[:, 0]], xy[cv[:, 2]] - xy[cv[:, 0]]
    area = 0.5 * np.abs(e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0])
    rng = np.random.default_rng(seed)
    c = rng.choice(len(cv), n, p=area / area.sum())
    w = rng.dirichlet([1, 1, 1], n)
    return (w[:, :, None] * xy[cv[c]]).sum(1)


def timed(fn, reps=3):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return out, 1e3 * float(np.median(ts))


def hbm(n_found, per_point, ms):
    return n_found * per_point / (ms * 1e-3) / HBM_PEAK


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--levels", type=int, default=8)
    ap.add_argument("--points", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    res = {"card": card(), "levels": a.levels}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)

    m = mesh(a.levels)
    s = solver(m)
    s.dev.set_solution(analytic(s))
    res.update(cells=int(m.n_cells), dofs=int(s.dofs.n))
    pts = random_points(m, a.points)
    (vals, cells), first_ms = timed(lambda: s.dev.evaluate(pts), 1)     # builds the index
    info = s.dev.points_index_info()
    res["index"] = dict(info, mean_bin=info["entries"] / max(info["nonempty_bins"], 1), first_call_ms=first_ms)
    found = int((cells >= 0).sum())
    (vals, cells), call_ms = timed(lambda: s.dev.evaluate(pts))
    k_ms = s.dev.time_kernel(8, a.reps)
    (_, grads, _), call_g_ms = timed(lambda: s.dev.evaluate(pts, gradients=True))
    kg_ms = s.dev.time_kernel(8, a.reps)
    res["random_points"] = dict(n=a.points, found=found, kernel_ms=k_ms, call_ms=call_ms, copies_and_host_ms=call_ms - k_ms,
                                kernel_grads_ms=kg_ms, call_grads_ms=call_g_ms, copies_and_host_grads_ms=call_g_ms - kg_ms,
                                points_per_s=found / (k_ms * 1e-3), hbm_fraction=hbm(found, BYTES_VALUES, k_ms),
                                hbm_fraction_grads=hbm(found, BYTES_VALUES + BYTES_GRADS, kg_ms))
    print(json.dumps(res), flush=True)

    if a.levels >= 1:
        src = solver(mesh(a.levels - 1))
        src.dev.set_solution(analytic(src))
        _, transfer_ms = timed(lambda: s.set_solution_from(src), 1)      # builds the source's index, then as below
        _, transfer_ms = timed(lambda: s.set_solution_from(src), 1)
        n_pts = s.part.n_own                                              # every owned support point of the fine mesh
        tk_ms = src.dev.time_kernel(8, 3)
        sidx = src.dev.points_index_info()
        res["transfer"] = dict(source_cells=int(src.mesh.n_cells), support_points=int(n_pts), kernel_ms=tk_ms, call_ms=transfer_ms,
                               copies_and_host_ms=transfer_ms - tk_ms, hbm_fraction=hbm(n_pts, BYTES_VALUES, tk_ms),
                               source_index=sidx)
    print(json.dumps(res), flush=True)
    out = os.environ.get("POINT_EVAL_OUT")
    if out:
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
