"""NavierStokesSolver — Python mirror of the reference class interface
(/root/reference src/NavierStokesSolver.hpp:407-795, src/NavierStokesSolver.cpp) driving the
B200 path: setup() -> topology (libnst.so) + one-time uploads; assemble_system(), solve_system(),
solve_newton(), solve(), output() keep the reference's names, order of operations, tolerances and
printed quantities; the Trilinos objects are the device CSR / vectors behind include/nsg.h.

The reference hard-codes every parameter (SURVEY §5 "config / flags"); here they are
constructor keywords whose DEFAULTS are the reference's constants.
"""
import math
import os
import sys
from dataclasses import dataclass, field

import numpy as np

from .device import PRECOND_BLOCK_DIAGONAL, PRECOND_BLOCK_TRIANGULAR, PRECOND_IDENTITY, DeviceProblem
from .topology import Dofs, Mesh, Part

_PRECONDS = {"identity": PRECOND_IDENTITY, "block_diagonal": PRECOND_BLOCK_DIAGONAL,
             "block_triangular": PRECOND_BLOCK_TRIANGULAR}


@dataclass
class Parameters:
    mesh_path: str = "../mesh/correct_mesh_yt.msh"   # cpp:15
    surface_entity: int = -1                         # -1: all surfaces (SURVEY F5 for mesh2d.msh)
    refine_levels: int = 0
    nu: float = 0.001                                # hpp:703
    rho: float = 1.0                                 # hpp:706
    p_out: float = 10.0                              # hpp:709
    g: float = 0.0                                   # hpp:438
    u_m: float = 1.5                                 # hpp:473
    H: float = 0.41                                  # hpp:474
    inlet_y0: float = 0.0
    # InletVelocity multiplies by sin(pi*get_time()/8) and set_time() is never called
    # (SURVEY F3): "frozen" reproduces that (factor sin(0)=0); "live" uses the current time;
    # "constant" uses factor 1.
    inlet_time_mode: str = "frozen"
    neumann_id: int = 10                             # cpp:320
    inlet_id: int = 11                               # cpp:357
    wall_ids: tuple = (12, 13)                       # cpp:367-368
    clear_inlet_before_walls: bool = False           # cpp:364 has boundary_functions.clear() commented out
    # The reference imposes the FULL boundary value g on every Newton increment (cpp:375-376), so with g != 0
    # the boundary value of the iterate grows by g per Newton iteration (harmless as shipped: g == 0, SURVEY F3).
    # "reference" reproduces that; "consistent" imposes g - u^k so that the iterate attains g (SURVEY §7).
    increment_bc: str = "reference"
    use_mass: bool = True                            # implicit Euler terms, cpp:249-251,288-290
    newton_max_iters: int = 1000                     # cpp:593
    newton_tolerance: float = 1e-2                   # cpp:594
    gmres_max_iters: int = 100000                    # cpp:566
    gmres_rel_tol: float = 1e-2                      # cpp:566
    gmres_n_tmp_vectors: int = 30                    # deal.II AdditionalData default
    preconditioner: str = "identity"                 # cpp:570
    # Stokes path ids (cpp:472,511,520-521) and solver settings (cpp:537)
    stokes_neumann_id: int = 1
    stokes_inlet_id: int = 0
    stokes_wall_ids: tuple = (2, 3)
    stokes_max_iters: int = 2000
    stokes_rel_tol: float = 1e-6
    output_dir: str = ""                             # "" = no files (cpp:681-728 writes XDMF/HDF5)
    dirichlet_diag: int = 0                          # include/nsg.h nsg_params: 0 TrilinosWrappers rule, 1 keep a non-zero diagonal
    force_boundary_id: int = -1                      # >= 0: record drag/lift on this boundary after every time step (N3)
    probe_points: tuple = ()                         # (x, y) points: record (u_x, u_y, p) there after every time step
    extra: dict = field(default_factory=dict)


class NavierStokesSolver:
    dim = 2  # hpp:411

    def __init__(self, degree_velocity, degree_pressure, T, deltat, params=None, device=0, rank=0, world_size=1,
                 comm_unique_id=None, stream=None, verbose=True, gather_objects=None, dist=None):
        if (degree_velocity, degree_pressure) != (2, 1):
            raise ValueError("the B200 path implements the reference's P2-P1 Taylor-Hood pair (main.cpp:9-10)")
        self.T = float(T)
        self.deltat = float(deltat)
        self.prm = params or Parameters()
        self.device, self.rank, self.world_size = device, rank, world_size
        self._uid, self._stream = comm_unique_id, stream
        # P > 1: callable(obj) -> [obj of rank 0, ..., obj of rank P-1] (e.g. torch.distributed.all_gather_object), used
        # by output() so that rank 0 can describe every rank's heavy-data file in the one .xdmf
        self._gather_objects = gather_objects
        # P > 1: an initialised torch.distributed module; switches the Krylov all-reduces to the fused NVLink path and
        # provides the object gather of output()
        self._dist = dist
        if dist is not None and gather_objects is None:
            def _gather(obj):
                out = [None] * dist.get_world_size()
                dist.all_gather_object(out, obj)
                return out
            self._gather_objects = _gather
        self.verbose = verbose and rank == 0
        self.time = 0.0
        self.history = []        # (time_step, newton_iter, residual_norm, gmres_its)
        self.force_history = []  # (time, F_x, F_y) when Parameters.force_boundary_id >= 0
        self.probe_history = []  # (time, values (n, 3)) when Parameters.probe_points is not empty

    def pcout(self, *a, **k):
        if self.verbose:
            print(*a, **k)
            sys.stdout.flush()

    # ---- setup (cpp:4-176) --------------------------------------------------------------------
    def setup(self, mesh=None):
        prm = self.prm
        self.pcout("Initializing the mesh")
        if mesh is None:
            mesh = Mesh.read_msh(prm.mesh_path, prm.surface_entity)
            if prm.refine_levels:
                mesh = mesh.refine(prm.refine_levels)
        self.mesh = mesh
        self.pcout(f"  Number of elements = {mesh.n_cells}")
        self.pcout("-----------------------------------------------")
        self.pcout("Initializing the DoF handler")
        cell_part = mesh.partition_rcb(self.world_size) if self.world_size > 1 else None
        self.dofs = Dofs(mesh, self.world_size, cell_part)
        self.pcout("  Number of DoFs: ")
        self.pcout(f"    velocity = {self.dofs.n_u}")
        self.pcout(f"    pressure = {self.dofs.n_p}")
        self.pcout(f"    total    = {self.dofs.n}")
        self.pcout("-----------------------------------------------")
        self.pcout("  Initializing the linear system")
        self.part = Part(self.dofs, self.rank, patterns=False)   # the device builds the sparsity patterns (SURVEY 8f N4)
        self.dev = DeviceProblem(self.part, self.device, self._stream)
        if self.world_size > 1:
            self.dev.comm_init(self.rank, self.world_size, self._uid)
            if self._dist is not None:
                self.dev.enable_peer_allreduce(self._dist)
        self._push_params(stokes=False)
        return self

    def _push_params(self, stokes):
        p = self.prm
        self.dev.set_params(nu=p.nu, rho=p.rho, p_out=p.p_out, deltat=self.deltat, forcing=(0.0, -p.g),
                            neumann_id=p.stokes_neumann_id if stokes else p.neumann_id,
                            use_mass=1 if p.use_mass else 0, stokes=1 if stokes else 0, dirichlet_diag=p.dirichlet_diag)

    def _inlet(self):
        mode = self.prm.inlet_time_mode
        t = 0.0 if mode == "frozen" else self.time
        tf = 1.0 if mode == "constant" else math.sin(math.pi * t / 8.0)
        return {"u_m": self.prm.u_m, "H": self.prm.H, "y0": self.prm.inlet_y0, "time_factor": tf}

    def _dirichlet(self, stokes=False):
        p = self.prm
        inlet_id = p.stokes_inlet_id if stokes else p.inlet_id
        walls = p.stokes_wall_ids if stokes else p.wall_ids
        second = {} if (stokes or p.clear_inlet_before_walls) else {inlet_id: True}
        second.update({w: False for w in walls})
        # interpolate_boundary_values walks the whole mesh (cpp:351-373): with a frozen / constant inlet the list is the same in
        # every Newton iteration of every time step, so it is evaluated once per (path, inlet factor)
        inlet = self._inlet()
        key = (bool(stokes), inlet["time_factor"])
        cache = self.__dict__.setdefault("_dirichlet_cache", {})
        if key not in cache:
            gd, gv = self.dofs.dirichlet_values([{inlet_id: True}, second], inlet)
            cache.clear()
            cache[key] = self.part.localize_dirichlet(gd, gv)
        ld, lv = cache[key]
        if not stokes and p.increment_bc == "consistent" and len(ld):
            lv = lv - self.dev.get_solution()[ld]
        return ld, lv

    # ---- assemble_system (cpp:178-378) --------------------------------------------------------
    def assemble_system(self):
        self.pcout("===============================================")
        self.pcout("Assembling the system")
        self.dev.assemble()
        d, v = self._dirichlet()
        self.dev.apply_dirichlet(d, v)

    # ---- solve_system (cpp:561-588) -------------------------------------------------------------
    def solve_system(self):
        self.pcout("===============================================")
        self.pcout("Solving system...")
        its, res, _ = self.dev.solve(_PRECONDS[self.prm.preconditioner], self.prm.gmres_rel_tol, self.prm.gmres_max_iters,
                                     self.prm.gmres_n_tmp_vectors, target=0)
        self.pcout(f"   {its} GMRES iterations")
        return its

    # ---- Stokes initial guess (cpp:380-559; call site commented out in the reference) -----------
    def assemble_stokes_system(self):
        self.pcout("===============================================")
        self.pcout("Assembling the Stokes system")
        self._push_params(stokes=True)
        self.dev.assemble()
        d, v = self._dirichlet(stokes=True)
        self.dev.apply_dirichlet(d, v, into_solution=True)
        self._push_params(stokes=False)

    def solve_stokes_system(self):
        self.pcout("===============================================")
        self.pcout("Solving the Stokes system")
        its, res, _ = self.dev.solve(PRECOND_BLOCK_TRIANGULAR, self.prm.stokes_rel_tol, self.prm.stokes_max_iters,
                                     self.prm.gmres_n_tmp_vectors, target=1)
        self.pcout(f"  {its} GMRES iterations")
        self.output(0, 0.0)
        return its

    # ---- solve_newton (cpp:590-627) -------------------------------------------------------------
    def solve_newton(self, time_step=0):
        n_max, tol = self.prm.newton_max_iters, self.prm.newton_tolerance
        n_iter, residual_norm = 0, tol + 1
        while n_iter < n_max and residual_norm > tol:
            self.assemble_system()
            residual_norm = self.dev.residual_norm()
            self.pcout(f"  Newton iteration {n_iter}/{n_max} - ||r|| = {residual_norm:.6e}", end="")
            its = None
            if residual_norm > tol:
                its = self.solve_system()
                self.pcout("System solved!")
                self.dev.update_solution()
            else:
                self.pcout(" < tolerance")
            self.history.append((time_step, n_iter, residual_norm, its))
            n_iter += 1
        return n_iter

    # ---- solve (cpp:629-679) ----------------------------------------------------------------------
    def solve(self, stokes_init=False):
        self.pcout("===============================================")
        self.time = 0.0
        if stokes_init:  # the block the reference has commented out (cpp:636-644)
            self.pcout("Finding the initial condition")
            self.assemble_stokes_system()
            self.solve_stokes_system()
            self.pcout("-----------------------------------------------")
        else:
            self.pcout("Applying the initial condition")
            self.dev.set_solution(np.zeros(self.part.n_own))  # FunctionU0 == 0 (hpp:478-497)
            self.output(0, 0.0)
            self.pcout("-----------------------------------------------")
        time_step = 0
        while self.time < self.T - 0.5 * self.deltat:
            self.time += self.deltat
            time_step += 1
            self.dev.push_time_level()
            self.pcout(f"n = {time_step:3d}, t = {self.time:5f}")
            self.solve_newton(time_step)
            if self.prm.force_boundary_id >= 0:
                f = self.dev.boundary_force(self.prm.force_boundary_id)
                self.force_history.append((self.time, float(f[0]), float(f[1])))
            if len(self.prm.probe_points):
                self.probe_history.append((self.time, self.point_values(self.prm.probe_points)))
            self.output(time_step, self.time)
            self.pcout("")

    # ---- output (cpp:681-728): XDMF + raw binary heavy data (output.py; HDF5 is not in this image) + npz restart data ----
    def output(self, time_step, time):
        self.pcout("===============================================")
        if not self.prm.output_dir:
            return
        os.makedirs(self.prm.output_dir, exist_ok=True)
        name = f"output-{time_step:04d}"
        sol = self.dev.get_solution()
        np.savez(os.path.join(self.prm.output_dir, f"{name}.rank{self.rank}.npz"), time=time, solution=sol,
                 l2g=self.part.l2g[: self.part.n_own], partitioning=self.rank)
        # XDMF + raw binary heavy data, one patch per owned cell as DataOut::build_patches makes them (cpp:685-727)
        from . import output as xout
        patches = xout.cell_patches(self.part, self.dev.get_solution_ghosted(), self.rank)
        layout = xout.write_rank_file(self.prm.output_dir, name, self.rank, patches)
        layouts = {self.rank: layout}
        if self.world_size > 1 and self._gather_objects is not None:
            layouts = {r: lay for r, lay in enumerate(self._gather_objects(layout))}
        if self.rank == 0:
            xout.write_xdmf(self.prm.output_dir, name, time, layouts)

    # ---- N3: drag / lift on the cylinder (boundary id 13, cpp:368); not in the reference ----------------
    def drag_lift(self, boundary_id=13, u_mean=1.0, diameter=0.1):
        """Force (F_x, F_y) and the coefficients 2F/(rho U^2 D)."""
        f = self.dev.boundary_force(boundary_id)
        return f, 2.0 * f / (self.prm.rho * u_mean ** 2 * diameter)

    # ---- point evaluation: probes, the pressure difference across the cylinder, transfer to another mesh ---------------
    def point_values(self, points):
        """(u_x, u_y, p) of the current solution at points (n, 2); NaN where no cell contains a point. With P > 1 every
        rank must pass the same points and gets the same values."""
        return self.dev.evaluate(np.asarray(points, np.float64).reshape(-1, 2))[0]

    def pressure_difference(self, front=(-0.5, 0.0), back=(0.5, 0.0)):
        """p(front) - p(back): the DFG cylinder benchmark's delta p (the repository's meshes: cylinder of radius 0.5 at
        the origin)."""
        v = self.point_values([front, back])
        return float(v[0, 2] - v[1, 2])

    def set_solution_from(self, source):
        """Interpolate the solution of another solver (e.g. on a coarser mesh of the same domain) at this solver's support
        points and make it the current solution (deal.II's VectorTools::interpolate_to_different_mesh). P = 1 only."""
        if self.world_size > 1 or source.world_size > 1:
            raise NotImplementedError("set_solution_from: transfer between partitioned meshes is not implemented")
        own = np.asarray(self.part.l2g[: self.part.n_own])
        xy = self.dofs.support_points()[own]
        vals, cells = source.dev.evaluate(xy)
        if (cells < 0).any():
            bad = np.flatnonzero(cells < 0)
            raise ValueError(f"{len(bad)} support points lie outside the source mesh (first at {xy[bad[0]].tolist()})")
        comp = np.where(own < self.dofs.n_u, own % 2, 2)
        self.dev.set_solution(vals[np.arange(len(own)), comp])

    # ---- helpers ----------------------------------------------------------------------------------
    def gather_solution(self):
        """Owned solution entries scattered into a global-size vector (zeros elsewhere)."""
        out = np.zeros(self.dofs.n)
        out[self.part.l2g[: self.part.n_own]] = self.dev.get_solution()
        return out
