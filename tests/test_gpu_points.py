"""-m gpu: point location and evaluation of the solution (nsg_eval_points, DeviceProblem.evaluate and the solver's probes,
pressure difference and solution transfer), against a numpy restatement that tests every cell for every point."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import meshgen
from conftest import ROOT, analytic_state, mesh_path

TOL = 1e-12   # barycentric tolerance of the containment test (same as the device)


# ---- numpy restatement --------------------------------------------------------------------------------------------------
def grad_lambda(xy, cv):
    """(T, 3, 2) gradients of the barycentric coordinates, from J^-T as the device's geometry kernel forms it."""
    x0 = xy[cv[:, 0]]
    J00, J01 = xy[cv[:, 1], 0] - x0[:, 0], xy[cv[:, 2], 0] - x0[:, 0]
    J10, J11 = xy[cv[:, 1], 1] - x0[:, 1], xy[cv[:, 2], 1] - x0[:, 1]
    det = J00 * J11 - J01 * J10
    a00, a01, a10, a11 = J11 / det, -J10 / det, -J01 / det, J00 / det
    return np.stack([np.stack([-(a00 + a01), -(a10 + a11)], 1), np.stack([a00, a10], 1), np.stack([a01, a11], 1)], 1)


def bary(xy, cv, gl, cells, pts):
    d = pts - xy[cv[cells, 0]]
    l1 = gl[cells, 1, 0] * d[..., 0] + gl[cells, 1, 1] * d[..., 1]
    l2 = gl[cells, 2, 0] * d[..., 0] + gl[cells, 2, 1] * d[..., 1]
    return np.stack([1.0 - l1 - l2, l1, l2], -1)


def np_locate(xy, cv, pts, gid=None, owned=None, chunk=128):
    """Global id of the owned cell of smallest global id whose barycentric coordinates are all >= -TOL (-1: none), and its
    local index; brute force over every cell."""
    T = len(cv)
    gid = np.arange(T) if gid is None else np.asarray(gid, np.int64)
    owned = np.ones(T, bool) if owned is None else np.asarray(owned).astype(bool)
    gl = grad_lambda(xy, cv)
    allc = np.arange(T)
    big = np.iinfo(np.int64).max
    best = np.full(len(pts), -1, np.int64)
    loc = np.full(len(pts), -1, np.int64)
    for s in range(0, len(pts), chunk):
        p = pts[s:s + chunk]
        with np.errstate(invalid="ignore"):
            lam = bary(xy, cv, gl, allc[None, :], p[:, None, :])
            inside = (lam >= -TOL).all(-1) & owned[None, :]
        key = np.where(inside, gid[None, :], big)
        k = key.argmin(1)
        hit = key[np.arange(len(p)), k] != big
        best[s:s + chunk] = np.where(hit, gid[k], -1)
        loc[s:s + chunk] = np.where(hit, k, -1)
    return best, loc


def np_eval(xy, cv, cd, sol, pts, loc):
    """values (n, 3) and grads (n, 2, 3) of the P2-P1 field in cell loc (NaN where loc < 0)."""
    n = len(pts)
    vals, grads = np.full((n, 3), np.nan), np.full((n, 2, 3), np.nan)
    ok = loc >= 0
    c, p = loc[ok], pts[ok]
    gl = grad_lambda(xy, cv)[c]
    l = bary(xy, cv, grad_lambda(xy, cv), c, p)
    l0, l1, l2 = l[:, 0], l[:, 1], l[:, 2]
    psi = np.stack([l0 * (2 * l0 - 1), l1 * (2 * l1 - 1), l2 * (2 * l2 - 1), 4 * l0 * l1, 4 * l1 * l2, 4 * l2 * l0], 1)
    uix = np.array([0, 3, 6, 9, 11, 13])
    ux, uy, pp = sol[cd[c][:, uix]], sol[cd[c][:, uix + 1]], sol[cd[c][:, [2, 5, 8]]]
    v = np.zeros((len(c), 3))
    g = np.zeros((len(c), 2, 3))
    for k in range(6):
        v[:, 0] += psi[:, k] * ux[:, k]
        v[:, 1] += psi[:, k] * uy[:, k]
    v[:, 2] = pp[:, 0] * l0 + pp[:, 1] * l1 + pp[:, 2] * l2
    for j in range(2):
        d0, d1, d2 = gl[:, 0, j], gl[:, 1, j], gl[:, 2, j]
        dpsi = [(4 * l0 - 1) * d0, (4 * l1 - 1) * d1, (4 * l2 - 1) * d2, 4 * (l0 * d1 + l1 * d0), 4 * (l1 * d2 + l2 * d1),
                4 * (l2 * d0 + l0 * d2)]
        for k in range(6):
            g[:, j, 0] += dpsi[k] * ux[:, k]
            g[:, j, 1] += dpsi[k] * uy[:, k]
        g[:, j, 2] = pp[:, 0] * d0 + pp[:, 1] * d1 + pp[:, 2] * d2
    vals[ok], grads[ok] = v, g
    return vals, grads


def part_arrays(part):
    return (np.asarray(part.xy).reshape(-1, 2), np.asarray(part.cell_vertices).reshape(-1, 3),
            np.asarray(part.cell_dofs).reshape(-1, 15))


def probe_points(mesh, rng, n_random=2000):
    """random points over the bounding box, every vertex, every edge midpoint, a random point on every edge (shared and
    boundary), the two cylinder points and points outside the domain."""
    xy, ev = mesh.xy, mesh.edge_vertices
    lo, hi = xy.min(0), xy.max(0)
    t = rng.random((len(ev), 1))
    return np.concatenate([lo + (hi - lo) * rng.random((n_random, 2)), xy, 0.5 * (xy[ev[:, 0]] + xy[ev[:, 1]]),
                           xy[ev[:, 0]] + t * (xy[ev[:, 1]] - xy[ev[:, 0]]),
                           [[-0.5, 0.0], [0.5, 0.0], [1e3, 1e3], [-1e3, 0.0], [lo[0] - 1e-3, lo[1]], [np.nan, 0.0],
                            [0.0, np.inf]]])


def rel_close(a, b, tol, scale=None):
    """|a - b| <= tol * scale, scale = max |b| of each component over all points (NaN where b is NaN)."""
    a, b = np.asarray(a).reshape(len(a), -1), np.asarray(b).reshape(len(b), -1)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    m = ~np.isnan(b)
    if scale is None:
        scale = np.where(m, np.abs(b), 0.0).max(0)
    err = np.where(m, np.abs(a - b), 0.0)
    assert (err <= tol * np.maximum(scale, 1e-300)).all(), (err.max(0), np.max(scale))


def term_scale(xy, cv, cd, sol, pts, loc):
    """Per point and gradient component: the sum of the magnitudes of the terms the gradient adds up (the scale of its rounding
    error, which on sliver cells, where grad lambda is large, far exceeds the largest gradient)."""
    n = len(pts)
    out = np.zeros((n, 6))
    ok = loc >= 0
    c = loc[ok]
    gl = np.abs(grad_lambda(xy, cv)[c])
    l = np.abs(bary(xy, cv, grad_lambda(xy, cv), c, pts[ok]))
    uix = np.array([0, 3, 6, 9, 11, 13])
    for j in range(2):
        dpsi = np.stack([(4 * l[:, 0] + 1) * gl[:, 0, j], (4 * l[:, 1] + 1) * gl[:, 1, j], (4 * l[:, 2] + 1) * gl[:, 2, j],
                         4 * (l[:, 0] * gl[:, 1, j] + l[:, 1] * gl[:, 0, j]), 4 * (l[:, 1] * gl[:, 2, j] + l[:, 2] * gl[:, 1, j]),
                         4 * (l[:, 2] * gl[:, 0, j] + l[:, 0] * gl[:, 2, j])], 1)
        out[ok, 2 * j] = (dpsi * np.abs(sol[cd[c][:, uix]])).sum(1)
        out[ok, 2 * j + 1] = (dpsi * np.abs(sol[cd[c][:, uix + 1]])).sum(1)
        out[ok, 4 + j] = (gl[:, :, j] * np.abs(sol[cd[c][:, [2, 5, 8]]])).sum(1)
    return out


def device_problem(pkg, mesh):
    d = pkg.Dofs(mesh)
    part = pkg.Part(d, 0)      # host-built patterns: the device pattern builder stops at valence 34, the wheel has 64
    return d, part, pkg.DeviceProblem(part, 0)


MESHES = {
    "square": lambda pkg: pkg.Mesh.read_msh(mesh_path("square_h0.1.msh")),
    "cmy": lambda pkg: pkg.Mesh.read_msh(mesh_path("cylinder_cmy.msh")),
    "mesh2d": lambda pkg: pkg.Mesh.read_msh(mesh_path("cylinder_mesh2d.msh"), 5),
    "wheel64": lambda pkg: meshgen.wheel(pkg, 64, 3),   # the largest valence nsg_set_mesh accepts (65 is refused)
    "bowtie": lambda pkg: meshgen.bowtie(pkg),
    "delaunay": lambda pkg: meshgen.delaunay(pkg, 1000, seed=3),
}


# ---- 1. exactness: P2 reproduces a quadratic velocity, P1 a linear pressure --------------------------------------------
def quadratic_field(p):
    x, y = p[..., 0], p[..., 1]
    v = np.stack([0.3 + 1.1 * x - 0.7 * y + 0.5 * x * x - 0.9 * x * y + 0.25 * y * y,
                  -0.2 + 0.4 * x + 0.8 * y - 0.6 * x * x + 0.35 * x * y - 0.15 * y * y, 1.5 - 2.0 * x + 0.75 * y], -1)
    g = np.stack([np.stack([1.1 + x - 0.9 * y, 0.4 - 1.2 * x + 0.35 * y, np.full_like(x, -2.0)], -1),
                  np.stack([-0.7 - 0.9 * x + 0.5 * y, 0.8 + 0.35 * x - 0.3 * y, np.full_like(x, 0.75)], -1)], -2)
    return v, g   # values (n, 3), grads (n, 2, 3): grads[i, d, k] = d(value k) / dx_d


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["square", "cmy"])
def test_interpolant_of_quadratic_field_is_exact(pkg, name):
    m = MESHES[name](pkg)
    d, part, dev = device_problem(pkg, m)
    sp = d.support_points()
    v, _ = quadratic_field(sp)
    comp = np.where(np.arange(d.n) < d.n_u, np.arange(d.n) % 2, 2)
    dev.set_solution(v[np.arange(d.n), comp][np.asarray(part.l2g[: part.n_own])])
    rng = np.random.default_rng(1)
    xy, cv = m.xy, m.cells
    c = rng.integers(0, m.n_cells, 2000)
    w = rng.dirichlet([1, 1, 1], 2000)
    pts = (w[:, :, None] * xy[cv[c]]).sum(1)
    vals, grads, cells = dev.evaluate(pts, gradients=True)
    assert (cells >= 0).all()
    ve, ge = quadratic_field(pts)
    rel_close(vals, ve, 1e-12)
    rel_close(grads, ge, 1e-12)
    dev.close()


# ---- 2. against the numpy restatement --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MESHES))
def test_matches_numpy_restatement(pkg, name):
    m = MESHES[name](pkg)
    d, part, dev = device_problem(pkg, m)
    xy, cv, cd = part_arrays(part)
    sol = analytic_state(d)[np.asarray(part.l2g)]
    dev.set_solution(sol[: part.n_own])
    pts = probe_points(m, np.random.default_rng(2))
    vals, grads, cells = dev.evaluate(pts, gradients=True)
    best, loc = np_locate(xy, cv, pts)
    assert np.array_equal(cells, best)
    assert (cells[-3:] == -1).all() and np.isnan(vals[-3:]).all() and np.isnan(grads[-3:]).all()   # outside, NaN, inf
    assert (cells[len(pts) - 7 - len(m.edge_vertices):] >= 0).sum() >= len(m.edge_vertices)    # points on edges are found
    v_np, g_np = np_eval(xy, cv, cd, sol, pts, loc)
    rel_close(vals, v_np, 1e-13)
    # gradients: 1e-13 of the largest one; on the Delaunay mesh's sliver cells the sum of the terms is the rounding scale
    scale = np.maximum(term_scale(xy, cv, cd, sol, pts, loc), np.nanmax(np.abs(g_np).reshape(len(pts), -1), 0))
    rel_close(grads, g_np, 1e-13, scale if name == "delaunay" else None)
    # the index: built by the first call, bounded bins
    info = dev.points_index_info()
    assert info["entries"] >= m.n_cells and info["max_bin"] >= 1 and info["bytes"] == 8 * (info["bins_x"] * info["bins_y"] + 1) + 4 * info["entries"]
    dev.close()


# ---- 3. transfer to a refined mesh ---------------------------------------------------------------------------------------
def _solver(pkg, mesh):
    s = pkg.NavierStokesSolver(2, 1, 0.05, 0.05, pkg.Parameters(), verbose=False)
    return s.setup(mesh)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["square", "cmy"])
def test_transfer_to_refined_mesh(pkg, name):
    m = MESHES[name](pkg)
    src = _solver(pkg, m)
    src.dev.set_solution(analytic_state(src.dofs)[np.asarray(src.part.l2g[: src.part.n_own])])
    dst = _solver(pkg, m.refine(1))     # red refinement, no boundary snap: the coarse P2 space is contained in the fine one
    dst.set_solution_from(src)
    rng = np.random.default_rng(4)
    c = rng.integers(0, m.n_cells, 3000)
    pts = (rng.dirichlet([1, 1, 1], 3000)[:, :, None] * m.xy[m.cells[c]]).sum(1)
    a, b = src.dev.evaluate(pts)[0], dst.dev.evaluate(pts)[0]
    rel_close(b, a, 1e-12)
    same = _solver(pkg, m)              # transfer to the same mesh reproduces the vector
    same.set_solution_from(src)
    x, y = same.dev.get_solution(), src.dev.get_solution()
    assert np.abs(x - y).max() <= 1e-13 * np.abs(y).max()
    for s in (src, dst, same):
        s.dev.close()


# ---- 4. ownership: the per-rank contexts of a partition on one GPU, combined on the host, are bitwise P = 1 ----------------
@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_partition_contexts_on_one_gpu_are_bitwise_one_rank(pkg, world):
    m = MESHES["cmy"](pkg)
    pts = probe_points(m, np.random.default_rng(5))
    pts = np.concatenate([pts, [[-0.5, -2.31253069e-09], [0.5, 2.31253069e-09]]])
    d1, p1, dev1 = device_problem(pkg, m)
    dev1.set_solution(analytic_state(d1)[np.asarray(p1.l2g[: p1.n_own])])
    ref = dev1.evaluate(pts, gradients=True)
    cp = m.partition_rcb(world)
    d = pkg.Dofs(m, world, cp)
    sol = analytic_state(d)
    best = np.full(len(pts), np.iinfo(np.int64).max)
    vals, grads = np.full((len(pts), 3), np.nan), np.full((len(pts), 2, 3), np.nan)
    finders = np.zeros(len(pts), np.int64)   # ranks that report a cell for the point
    in_ghost = 0                             # points that only a ghost cell of a rank contains: the owned filter decides
    for r in range(world):
        part = pkg.Part(d, r, patterns=False)
        dev = pkg.DeviceProblem(part, 0)
        dev.set_solution_ghosted(sol[np.asarray(part.l2g)])
        v, g, c = dev.evaluate(pts, gradients=True, collective=False)
        xy, cv, _ = part_arrays(part)
        any_local, _ = np_locate(xy, cv, pts, gid=part.cell_ids)   # every local cell, ghosts included
        in_ghost += int(((any_local >= 0) & (c < 0)).sum())
        assert (cp[c[c >= 0]] == r).all()   # a rank answers from its owned cells only, never from a ghost cell
        finders += c >= 0
        take = (c >= 0) & (c < best)
        best[take], vals[take], grads[take] = c[take], v[take], g[take]
        dev.close()
    assert in_ghost > 0
    # some rank answers where P = 1 finds a cell (two or more on a rank interface, each from its own owned cell), none elsewhere
    assert np.array_equal(finders > 0, ref[2] >= 0)
    cells = np.where(best == np.iinfo(np.int64).max, -1, best)
    assert np.array_equal(cells, ref[2])
    assert np.array_equal(vals.view(np.uint64), ref[0].view(np.uint64))
    assert np.array_equal(grads.view(np.uint64), np.ascontiguousarray(ref[1]).view(np.uint64))
    dev1.close()


# ---- 5. collective mode on P GPUs ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_collective_mode_is_bitwise_one_rank(world, tmp_path):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(29633 + world), os.path.join(ROOT, "scripts", "points_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, POINTS_RESULT_DIR=str(tmp_path)))
    assert out.returncode == 0, f"{out.stdout[-2000:]}\n{out.stderr[-2000:]}"
    for r in range(world):
        path = tmp_path / f"rank{r}.json"
        assert path.exists(), f"rank {r} wrote no result\n{out.stdout[-2000:]}\n{out.stderr[-2000:]}"
        res = json.loads(path.read_text())
        assert res["world"] == world and res["n_points"] > 1000
        assert res["cells_equal"] and res["values_bitwise"] and res["grads_bitwise"], res
        assert res["probe_history_equal"], res


# ---- 6. solver level: probes and the pressure difference ---------------------------------------------------------------
@pytest.mark.gpu
def test_probes_and_pressure_difference_in_a_short_run(pkg):
    import dataclasses
    from oracle.oracle import Oracle
    probes = ((-0.5, 0.0), (0.5, 0.0), (2.0, 0.5), (8.0, -1.0))
    prm = pkg.Parameters(mesh_path=mesh_path("cylinder_mesh2d.msh"), surface_entity=5, nu=0.05, u_m=1.5, H=4.1, inlet_y0=-2.0,
                         inlet_time_mode="constant", preconditioner="identity", force_boundary_id=3, p_out=0.0,
                         increment_bc="consistent", neumann_id=1, inlet_id=0, wall_ids=(2, 3), newton_max_iters=8,
                         gmres_rel_tol=1e-12, gmres_max_iters=1000000, probe_points=probes)
    mesh = pkg.Mesh.read_msh(prm.mesh_path, prm.surface_entity)
    mesh.tag_boundary_box(0, 1, 2, 3)
    s = pkg.NavierStokesSolver(2, 1, 0.1, 0.05, prm, verbose=False)
    s.setup(mesh)
    after_step = []
    s.output = lambda step, t: after_step.append(s.dev.evaluate(np.array(probes))[0]) if step else None
    o = pkg.NavierStokesSolver(2, 1, 0.1, 0.05, dataclasses.replace(prm, probe_points=()), verbose=False)
    o.mesh, o.dofs = s.mesh, s.dofs
    o.part = pkg.Part(s.dofs, 0)
    o.dev = Oracle(o.part)
    o._push_params(stokes=False)
    s.solve()
    o.solve()
    assert len(s.probe_history) == len(after_step) == 2
    for (t, v), w, tt in zip(s.probe_history, after_step, (0.05, 0.1)):
        assert abs(t - tt) < 1e-12 and np.array_equal(v, w) and not np.isnan(v).any()
    xy, cv, cd = part_arrays(o.part)
    xo = o.dev.get_solution()
    pts = np.array([[-0.5, 0.0], [0.5, 0.0]])
    _, loc = np_locate(xy, cv, pts)
    v_np, _ = np_eval(xy, cv, cd, xo, pts, loc)
    dp_np = v_np[0, 2] - v_np[1, 2]
    dp = s.pressure_difference()
    assert dp == s.probe_history[-1][1][0, 2] - s.probe_history[-1][1][1, 2]
    assert abs(dp - dp_np) <= 1e-8 * np.abs(xo[s.dofs.n_u:]).max(), (dp, dp_np)
    assert abs(dp) > 1e-3
    s.dev.close()


# ---- 7. error paths -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_error_paths(pkg):
    import ctypes as C
    lib = importlib.import_module("navier-stokes-dealii_b200._lib")
    L = lib.nsg()
    h = C.c_void_p()
    lib.nsg_check(L.nsg_create(0, C.byref(h)))
    pts, vals = np.zeros(2), np.zeros(3)
    assert L.nsg_eval_points(h, 1, pts, 0, vals, None, None) == -5        # NSG_ERR_STATE: no mesh yet
    L.nsg_destroy(h)
    m = MESHES["square"](pkg)
    d, part, dev = device_problem(pkg, m)
    with pytest.raises(lib.NsgError):                                     # the index does not exist before the first call
        dev.points_index_info()
    v, c = dev.evaluate(np.zeros((0, 2)))                                 # n = 0: nothing to do
    assert v.shape == (0, 3) and c.shape == (0,)
    with pytest.raises(lib.NsgError):
        dev.points_index_info()
    with pytest.raises(ValueError):
        dev.evaluate(np.zeros((5, 3)))
    with pytest.raises(ValueError):
        dev.evaluate(np.zeros(6))
    with pytest.raises(ValueError):
        dev.set_solution_ghosted(np.zeros(part.n_loc + 1))
    s = pkg.NavierStokesSolver(2, 1, 0.05, 0.05, pkg.Parameters(), world_size=2, verbose=False)
    with pytest.raises(NotImplementedError):
        s.set_solution_from(s)
    dev.close()
