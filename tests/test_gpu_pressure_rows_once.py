"""-m gpu: the pressure rows of J and the pressure mass matrix Mp are integrated once and kept across assemblies.

They depend on the geometry and nu only, so nsg_assemble integrates them in the first call and again only after something
changed them: a new nu, a Dirichlet list that constrains a pressure row, a switch of the assembly variant.  Every test here
holds one DeviceProblem through a sequence of calls and compares J, Mp and R after each assembly BITWISE with a fresh
DeviceProblem that did a single assembly (plus the same Dirichlet list, where the sequence applies one) with the same state,
parameters and variant.  A missed invalidation leaves stale pressure rows behind and fails the comparison.  The flag lives in
the device context, so there is no CPU part."""
import os

import numpy as np
import pytest

import meshgen as mg
from conftest import GOLDEN, analytic_state

pytestmark = pytest.mark.gpu

PARAMS = dict(rho=1.3, p_out=10.0, deltat=0.05, forcing=(0.0, -0.7), use_mass=1, stokes=0)
NU, NU2 = 0.001, 0.0025

# name -> (mesh builder, Neumann id, Dirichlet calls, inlet data)
MESHES = {
    "square_h0.1": (lambda pkg: pkg.Mesh.read_msh(os.path.join(GOLDEN, "square_h0.1.msh")), 1,
                    [{0: True}, {2: False, 3: False}], dict(u_m=1.5, H=1.0)),
    "delaunay3000": (lambda pkg: mg.delaunay(pkg, 3000), mg.NEUMANN, mg.CALLS, mg.INLET),
}
_BUILT = {}


class Case:
    def __init__(self, pkg, name):
        build, self.neumann, calls, inlet = MESHES[name]
        self.pkg = pkg
        self.d = pkg.Dofs(build(pkg))
        self.part = pkg.Part(self.d, 0)
        self.gd, self.gv = self.d.dirichlet_values(calls, dict(time_factor=1.0, **inlet))
        assert (self.gd < self.part.n_own_u).all(), "the inlet list constrains velocity rows only"

    def params(self, nu):
        return dict(PARAMS, nu=nu, neumann_id=self.neumann)

    def device(self, variant, nu):
        dev = self.pkg.DeviceProblem(self.part, 0)
        dev.set_tuning(1, variant)
        dev.set_params(**self.params(nu))
        return dev

    def fresh(self, variant, nu, sol, sol_old, dirichlet=None):
        """J, Mp, R of a new DeviceProblem after one assembly (and the Dirichlet list, if given)."""
        dev = self.device(variant, nu)
        dev.set_solution(sol)
        dev.set_solution_old(sol_old)
        dev.assemble()
        if dirichlet is not None:
            dev.apply_dirichlet(*dirichlet)
        out = state_of(dev)
        dev.close()
        return out


def case(pkg, name):
    if name not in _BUILT:
        _BUILT[name] = Case(pkg, name)
    return _BUILT[name]


def state_of(dev):
    return dev.get_matrix_values(), dev.get_pm_values(), dev.get_residual()


def assert_bitwise(got, want, what):
    for a, b, label in zip(got, want, ("J", "Mp", "R")):
        assert np.array_equal(a.view(np.int64), b.view(np.int64)), f"{what}: {label} differs from a fresh assembly in {int((a != b).sum())} entries"


def assemble_and_check(c, dev, variant, nu, sol, sol_old, what):
    dev.set_solution(sol)
    dev.set_solution_old(sol_old)
    dev.assemble()
    assert_bitwise(state_of(dev), c.fresh(variant, nu, sol, sol_old), what)


CASES = [(name, v) for name in MESHES for v in (0, 4, 5)]


@pytest.mark.parametrize("name,variant", CASES)
def test_newton_steps(pkg, name, variant):
    """assemble, apply_dirichlet, solve, new solution, assemble again - four times."""
    c = case(pkg, name)
    dev = c.device(variant, NU)
    sol, sol_old = analytic_state(c.d), analytic_state(c.d, 0.9)
    for k in range(4):
        assemble_and_check(c, dev, variant, NU, sol, sol_old, f"step {k}")
        dev.apply_dirichlet(c.gd, c.gv)
        assert_bitwise(state_of(dev), c.fresh(variant, NU, sol, sol_old, (c.gd, c.gv)), f"step {k} after Dirichlet")
        dev.solve(0, 1e-2, 200, 30, 0, check=False)
        sol = sol + dev.get_delta()
    dev.close()


@pytest.mark.parametrize("name,variant", CASES)
def test_viscosity_change_and_back(pkg, name, variant):
    c = case(pkg, name)
    dev = c.device(variant, NU)
    sol, sol_old = analytic_state(c.d), analytic_state(c.d, 0.9)
    assemble_and_check(c, dev, variant, NU, sol, sol_old, "nu")
    dev.set_params(**c.params(NU))  # the same parameters again
    assemble_and_check(c, dev, variant, NU, sol, sol_old, "nu set again")
    dev.set_params(**c.params(NU2))
    assemble_and_check(c, dev, variant, NU2, sol, sol_old, "new nu")
    dev.set_params(**c.params(NU))
    assemble_and_check(c, dev, variant, NU, sol, sol_old, "nu back")
    dev.close()


@pytest.mark.parametrize("name,variant", CASES)
def test_pressure_dirichlet_then_plain_assembly(pkg, name, variant):
    """A list that constrains pressure rows rewrites them (cleared rows, reset diagonals); the next assembly without those rows
    must bring back B and the zero p-p block."""
    c = case(pkg, name)
    n_u, n_p = c.part.n_own_u, c.part.n_own_p
    pdofs = n_u + np.array([0, n_p // 3, n_p - 1])
    gd = np.concatenate([c.gd, pdofs]).astype(np.int32)
    gv = np.concatenate([c.gv, [0.5, -1.0, 2.0]])
    dev = c.device(variant, NU)
    sol, sol_old = analytic_state(c.d), analytic_state(c.d, 0.9)
    assemble_and_check(c, dev, variant, NU, sol, sol_old, "before")
    dev.apply_dirichlet(gd, gv)
    with_p = state_of(dev)
    assert_bitwise(with_p, c.fresh(variant, NU, sol, sol_old, (gd, gv)), "pressure Dirichlet")
    sol = sol + 0.01 * analytic_state(c.d, 0.5)
    assemble_and_check(c, dev, variant, NU, sol, sol_old, "assembly after the pressure Dirichlet")
    dev.apply_dirichlet(c.gd, c.gv)
    assert_bitwise(state_of(dev), c.fresh(variant, NU, sol, sol_old, (c.gd, c.gv)), "velocity Dirichlet after")
    dev.close()


@pytest.mark.parametrize("name,variant", CASES)
def test_block_preconditioned_solve_between_assemblies(pkg, name, variant):
    """The block preconditioners factorise ILU(0) copies of the velocity block and Mp; J and Mp themselves stay as assembled."""
    c = case(pkg, name)
    dev = c.device(variant, NU)
    sol, sol_old = analytic_state(c.d), analytic_state(c.d, 0.9)
    for precond in (pkg.PRECOND_BLOCK_TRIANGULAR, pkg.PRECOND_BLOCK_DIAGONAL):
        assemble_and_check(c, dev, variant, NU, sol, sol_old, f"before precond {precond}")
        dev.apply_dirichlet(c.gd, c.gv)
        dev.solve(precond, 1e-4, 200, 30, 0, check=False)
        sol = sol + dev.get_delta()
    assemble_and_check(c, dev, variant, NU, sol, sol_old, "after the block-preconditioned solves")
    dev.close()


@pytest.mark.parametrize("name", list(MESHES))
def test_variant_switch(pkg, name):
    """5 -> 0 -> 4 -> 5 -> 4 on one context; each assembly is bitwise what a fresh context of that variant gives."""
    c = case(pkg, name)
    sol, sol_old = analytic_state(c.d), analytic_state(c.d, 0.9)
    dev = c.device(5, NU)
    for variant in (5, 0, 4, 5, 4):
        dev.set_tuning(1, variant)
        assemble_and_check(c, dev, variant, NU, sol, sol_old, f"variant {variant}")
    dev.close()


@pytest.mark.parametrize("name,variant", CASES)
def test_launches_per_assembly(pkg, name, variant):
    """The first assembly launches the pressure-row kernel; the following ones launch exactly one kernel less, until nu
    changes."""
    c = case(pkg, name)
    dev = c.device(variant, NU)
    dev.set_solution(analytic_state(c.d))
    counts = []
    for nu in (NU, NU, NU, NU2, NU2):
        dev.set_params(**c.params(nu))
        before = dev.counters()["launches"]
        dev.assemble()
        counts.append(dev.counters()["launches"] - before)
    dev.close()
    full = counts[0]
    assert counts == [full, full - 1, full - 1, full, full - 1], counts
