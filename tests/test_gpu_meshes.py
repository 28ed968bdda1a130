"""-m gpu: the CUDA kernels on generated meshes (tests/meshgen.py) with what the shipped meshes lack - vertices of 9 to 65
cells, Jacobian rows of up to 458 entries, a vertex whose cells form two open fans, clockwise cells.  These run the fan tree's
steps 8 (valence >= 9) and 16 (valence >= 17) and a warp filled by one owner (valence 32), the SpMV tail loops past 64 entries
of a row, the ILU(0) solves on long rows, and the fallbacks of the assembly: variant 4 (the fan scheme refuses: mixed
orientation), variant 0 (valence 33-64) and the refusal beyond that.

Fallbacks are shown by bitwise equality: the default assembly must give exactly the bits of the variant it falls back to, and
differ from the other one (the variants sum in different orders)."""
import numpy as np
import pytest
import scipy.sparse as sp

import meshgen as mg
from conftest import analytic_state, row_scaled_err
from oracle.oracle import Oracle
from test_gpu_parity import check_path, set_path

pytestmark = pytest.mark.gpu

# name -> generator; the wheels have 3 rings (wheel32: 6, for the ILU level structure)
CASES = {
    "wheel9": lambda pkg: mg.wheel(pkg, 9, 3),
    "wheel16": lambda pkg: mg.wheel(pkg, 16, 3),
    "wheel31": lambda pkg: mg.wheel(pkg, 31, 3),
    "wheel32": lambda pkg: mg.wheel(pkg, 32, 6),
    "wheel33": lambda pkg: mg.wheel(pkg, 33, 3),
    "wheel34": lambda pkg: mg.wheel(pkg, 34, 3),
    "wheel35": lambda pkg: mg.wheel(pkg, 35, 3),
    "wheel65": lambda pkg: mg.wheel(pkg, 65, 3),
    "bowtie": lambda pkg: mg.bowtie(pkg),
    "delaunay3000": lambda pkg: mg.delaunay(pkg, 3000),
    "delaunay8000": lambda pkg: mg.delaunay(pkg, 8000),
}
_BUILT = {}


def case(pkg, name):
    if name not in _BUILT:
        m = CASES[name](pkg)
        d = pkg.Dofs(m)
        _BUILT[name] = (m, d, pkg.Part(d, 0))
    return _BUILT[name]


def serves(name, variant):
    """Assembly variants that serve the mesh: 5 and 4 up to valence 32, 0 up to 64."""
    k = int(name[5:]) if name.startswith("wheel") else 24 if name == "bowtie" else 16
    return k <= (64 if variant == 0 else 32)


PARAMS = dict(nu=0.001, rho=1.3, p_out=10.0, deltat=0.05, forcing=(0.0, -0.7), neumann_id=mg.NEUMANN)


def mode_params(mode):
    return dict(PARAMS, use_mass=0 if mode == "steady" else 1, stokes=1 if mode == "stokes" else 0)


def run_assembly(obj, d, mode, dirichlet=None):
    """J, Mp, R after assemble() (and J, R, |R| after apply_dirichlet when `dirichlet` = (dofs, values) is given)."""
    obj.set_params(**mode_params(mode))
    obj.set_solution(analytic_state(d))
    obj.set_solution_old(analytic_state(d, 0.9))
    obj.assemble()
    out = [obj.get_matrix_values(), obj.get_pm_values(), obj.get_residual()]
    if dirichlet is not None:
        obj.apply_dirichlet(*dirichlet, into_solution=(mode == "stokes"))
        out += [obj.get_matrix_values(), obj.get_residual(), obj.residual_norm()]
    return out


_ORACLE = {}


def oracle_assembly(pkg, name, mode):
    if (name, mode) not in _ORACLE:
        m, d, part = case(pkg, name)
        gd, gv = d.dirichlet_values(mg.CALLS, dict(time_factor=1.0, **mg.INLET))
        _ORACLE[name, mode] = run_assembly(Oracle(part), d, mode, (gd, gv))
    return _ORACLE[name, mode]


def assert_matches_oracle(got, want, part, tol=1e-12):
    Jd, Md, Rd, Jd2, Rd2, nd = got
    Jo, Mo, Ro, Jo2, Ro2, no = want
    assert row_scaled_err(Jd, Jo, part.jac_rowptr) <= tol
    assert row_scaled_err(Md, Mo, part.pm_rowptr) <= tol
    assert np.abs(Rd - Ro).max() <= tol * np.abs(Ro).max()
    assert row_scaled_err(Jd2, Jo2, part.jac_rowptr) <= tol
    assert np.abs(Rd2 - Ro2).max() <= tol * np.abs(Ro2).max()
    assert abs(nd - no) <= tol * no


def device_assembly(pkg, part, d, mode, variant=None, dirichlet=None):
    dev = pkg.DeviceProblem(part, 0)
    if variant is not None:
        dev.set_tuning(1, variant)
    out = run_assembly(dev, d, mode, dirichlet)
    dev.close()
    return out


ASM_CASES = ["wheel9", "wheel16", "wheel31", "wheel32", "wheel33", "wheel34", "bowtie", "delaunay3000"]


@pytest.mark.parametrize("name", ASM_CASES)
@pytest.mark.parametrize("mode", ["newton", "steady", "stokes"])
@pytest.mark.parametrize("variant", [0, 4, 5])
def test_assembly_against_oracle(pkg, name, mode, variant):
    """J and Mp to 1e-12 of the row maximum, R to 1e-12 of its maximum, before and after the Dirichlet rows (non-zero inlet
    data).  In Stokes mode two exact identities that a dropped or doubled fan cell breaks: the velocity rows annihilate a
    constant x-velocity, and Mp sums to area / nu."""
    if not serves(name, variant):
        pytest.skip(f"variant {variant} does not serve {name}")
    m, d, part = case(pkg, name)
    gd, gv = d.dirichlet_values(mg.CALLS, dict(time_factor=1.0, **mg.INLET))
    assert np.abs(gv).max() > 0.5
    got = device_assembly(pkg, part, d, mode, variant, (gd, gv))
    assert_matches_oracle(got, oracle_assembly(pkg, name, mode), part)
    if mode == "stokes":
        J = sp.csr_matrix((got[0], part.jac_col, part.jac_rowptr), shape=(d.n, d.n))
        ones = np.zeros(d.n)
        ones[0:d.n_u:2] = 1.0
        assert np.abs((J @ ones)[:d.n_u]).max() <= 1e-11 * np.abs(got[0]).max()
        xy, cv = m.xy, m.cells
        a, b, c = xy[cv[:, 0]], xy[cv[:, 1]], xy[cv[:, 2]]
        area = 0.5 * np.abs((b[:, 0] - a[:, 0]) * (c[:, 1] - a[:, 1]) - (c[:, 0] - a[:, 0]) * (b[:, 1] - a[:, 1])).sum()
        assert abs(got[1].sum() - area / PARAMS["nu"]) <= 1e-12 * area / PARAMS["nu"]


def longdouble_spmv(part, vals, x):
    rp = np.asarray(part.jac_rowptr)
    prod = np.asarray(vals, np.longdouble) * np.asarray(x, np.longdouble)[np.asarray(part.jac_col)]
    lens = np.diff(rp)
    y = np.zeros(len(lens), np.longdouble)
    nz = lens > 0
    y[nz] = np.add.reduceat(prod, rp[:-1][nz])
    return y


@pytest.mark.parametrize("name", ["wheel32", "wheel34", "delaunay3000", "delaunay8000"])
def test_spmv_against_longdouble(pkg, name):
    """Every row within (len + 2) 2^-53 (|J||x|)_i of the sum in extended precision: a single entry lost or added fails this
    bound, unlike a tolerance relative to max |y|.  Rows past 64 entries run the tail loops of variants 1, 4 and 7."""
    m, d, part = case(pkg, name)
    lens = mg.row_lengths(part)
    assert (lens > 64).sum() >= 3
    dev = pkg.DeviceProblem(part, 0)
    dev.set_params(**PARAMS)
    dev.set_solution(analytic_state(d, 0.3))
    dev.assemble()
    vals = dev.get_matrix_values()
    x = np.random.default_rng(11).standard_normal(d.n)
    y_ref = longdouble_spmv(part, vals, x)
    absy = sp.csr_matrix((np.abs(vals), part.jac_col, part.jac_rowptr), shape=(d.n, d.n)) @ np.abs(x)
    bound = (lens + 2) * 2.0 ** -53 * absy
    out = {}
    for variant in (0, 1, 4, 7):
        dev.set_tuning(0, variant)
        y = dev.spmv(x)
        err = np.abs(np.asarray(y, np.longdouble) - y_ref).astype(np.float64)
        bad = np.flatnonzero(err > bound)
        assert len(bad) == 0, (variant, bad[:5], lens[bad[:5]], err[bad[:5]], bound[bad[:5]])
        out[variant] = y
    assert np.array_equal(out[4], out[7])
    dev.close()


@pytest.mark.parametrize("name,parts", [("delaunay3000", 1), ("delaunay3000", 3), ("wheel32", 1), ("wheel32", 3)])
def test_device_pattern_long_rows(pkg, name, parts):
    """The pattern built on the device equals the host's bit for bit, whole mesh and every part of a 3-way partition, and
    assembly through either gives the same bits."""
    m = CASES[name](pkg)
    cp = m.partition_rcb(parts) if parts > 1 else None
    d = pkg.Dofs(m, parts, cp)
    for rank in range(parts):
        host = pkg.Part(d, rank)
        lean = pkg.Part(d, rank, patterns=False)
        dev_h, dev_d = pkg.DeviceProblem(host, 0), pkg.DeviceProblem(lean, 0)
        rp, col, prp, pcol = dev_d.get_pattern()
        assert np.array_equal(rp, host.jac_rowptr) and np.array_equal(col, host.jac_col)
        assert np.array_equal(prp, host.pm_rowptr) and np.array_equal(pcol, host.pm_col)
        sol = analytic_state(d)[host.l2g]
        out = []
        for dev in (dev_h, dev_d):
            dev.set_params(nu=0.01, neumann_id=mg.NEUMANN)
            dev.set_solution(sol[: host.n_own])
            dev.assemble()
            out.append((dev.get_matrix_values(), dev.get_pm_values(), dev.get_residual()))
            dev.close()
        for a, b in zip(*out):
            assert np.array_equal(a, b)


def test_device_pattern_refuses_valence_35(pkg):
    """An interior vertex of 35 cells has 106 velocity nodes in its patch, more than the builder's 104: the error states the
    builder's limit (34 inside the domain)."""
    m, d, part = case(pkg, "wheel35")
    with pytest.raises(Exception, match="valence <= 34"):
        pkg.DeviceProblem(pkg.Part(d, 0, patterns=False), 0)


def precond_system(pkg, name):
    m, d, part = case(pkg, name)
    gd, gv = d.dirichlet_values(mg.CALLS, dict(time_factor=1.0, **mg.INLET))
    dev, o = pkg.DeviceProblem(part, 0), Oracle(part)
    for obj in (dev, o):
        obj.set_params(nu=0.01, neumann_id=mg.NEUMANN)
        obj.set_solution(analytic_state(d, 0.05))
        obj.set_solution_old(analytic_state(d, 0.045))
        obj.assemble()
        obj.apply_dirichlet(gd, gv)
    return d, part, dev, o


@pytest.mark.parametrize("name", ["delaunay3000", "wheel32"])
def test_ilu_long_rows(pkg, name):
    """ILU(0) of both blocks with rows past 64 entries: the level-scheduled solves against the oracle, the single-launch and
    one-CTA solves bitwise equal to them over three right-hand sides."""
    d, part, dev, o = precond_system(pkg, name)
    for which, n in ((0, d.n_u), (1, d.n_p)):
        xs = [np.random.default_rng(17 + which + 10 * r).standard_normal(n) for r in range(3)]
        dev.set_tuning(4, 0)
        refs = [dev.ilu_apply(which, x) for x in xs]
        want = o.ilu_apply(which, xs[0])
        assert np.abs(refs[0] - want).max() <= 1e-11 * np.abs(want).max(), which
        for variant in (1, 2, -1):
            dev.set_tuning(4, variant)
            for x, ref in zip(xs, refs):
                assert np.array_equal(dev.ilu_apply(which, x), ref), (which, variant)
    dev.close()


@pytest.mark.parametrize("name", ["delaunay3000", "delaunay8000"])
def test_identity_gmres_fixed_steps(pkg, name):
    """84 GMRES(28) steps against the oracle, on the one-kernel path (27 022 unknowns) and on the multi-kernel path with and
    without CUDA graphs (72 022 unknowns; the two give the same bits).  The first restart cycle agrees to 1e-9.

    After the first restart the sliver cells along the hull show: on delaunay8000 the residual history right after the restart
    moves by up to 3e-7 when J is perturbed by one ulp at random, and a plain numpy GMRES(28) on the oracle's matrix differs
    from the oracle by 1.5e-5 (at step 35) - rounding amplified by ~1e11 whatever the kernels.  There the bound is 1e-4 for the
    history and 1e-5 of max |x| for the iterate (the one-ulp spread of the iterate is 9e-7); delaunay3000 keeps 1e-8."""
    m, d, part = case(pkg, name)
    paths = ("fused",) if d.n <= 65536 else ("graphs", "plain")
    tol_all, tol_x = (1e-8, 1e-8) if paths == ("fused",) else (1e-4, 1e-5)
    gd, gv = d.dirichlet_values(mg.CALLS, dict(time_factor=1.0, **mg.INLET))
    dev, o = pkg.DeviceProblem(part, 0), Oracle(part)
    for obj in (dev, o):
        obj.set_params(nu=0.01, neumann_id=mg.NEUMANN)
        obj.set_solution(analytic_state(d, 0.05))
        obj.set_solution_old(analytic_state(d, 0.045))
        obj.assemble()
        obj.apply_dirichlet(gd, gv)
    x0 = dev.get_delta()
    o.set_delta(x0)
    ro = o.solve(0, 1e-14, 84, 30, 0)
    h2, xo = o.gmres_history(), o.get_delta()
    assert ro[0] == 84 and ro[2] != 0
    out = []
    for path in paths:
        set_path(dev, path)
        dev.set_delta(x0)
        rd = dev.solve(0, 1e-14, 84, 30, 0, check=False)
        check_path(dev, path, None if path == "fused" else 7)
        assert rd[0] == 84 and rd[2] == -3
        h1, xd = dev.gmres_history(), dev.get_delta()
        assert np.abs(h1[:28] / h2[:28] - 1).max() <= 1e-9, path
        assert np.abs(h1 / h2 - 1).max() <= tol_all, path
        assert np.abs(xd - xo).max() <= tol_x * np.abs(xo).max(), path
        out.append((h1, xd))
    if len(out) == 2:
        assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    dev.close()


# ---- fallbacks -------------------------------------------------------------------------------------------------------------

def all_variants(pkg, part, d, mode="newton"):
    """Default assembly, then each explicitly selected variant on the same context (None where selecting it raises)."""
    dev = pkg.DeviceProblem(part, 0)
    out = {"default": run_assembly(dev, d, mode)}
    for v in (0, 4, 5):
        try:
            dev.set_tuning(1, v)
        except Exception as e:
            out[v] = str(e)
            continue
        out[v] = run_assembly(dev, d, mode)
    dev.close()
    return out


def same(a, b):
    return not isinstance(b, str) and all(np.array_equal(x, y) for x, y in zip(a, b))


def test_fallback_wheel32_takes_fan_and_variant4(pkg):
    """Valence 32: the fan scheme serves it by default (its head lane's fan fills a warp), and variant 4 serves it too."""
    m, d, part = case(pkg, "wheel32")
    out = all_variants(pkg, part, d)
    assert same(out["default"], out[5]) and not same(out["default"], out[4]) and not same(out["default"], out[0])
    want = oracle_assembly(pkg, "wheel32", "newton")
    for v in (0, 4, 5):
        assert row_scaled_err(out[v][0], want[0], part.jac_rowptr) <= 1e-12
        assert np.abs(out[v][2] - want[2]).max() <= 1e-12 * np.abs(want[2]).max()


@pytest.mark.parametrize("name", ["wheel33", "wheel34"])
def test_fallback_to_variant0(pkg, name):
    """Valence 33 and 34: neither the fan scheme nor variant 4 serves the mesh, the default assembly is variant 0's."""
    m, d, part = case(pkg, name)
    out = all_variants(pkg, part, d)
    assert same(out["default"], out[0])
    assert "valence <= 32" in out[5]
    assert f"has {name[5:]} incident cells" in out[4] and "at most 32" in out[4]
    gd, gv = d.dirichlet_values(mg.CALLS, dict(time_factor=1.0, **mg.INLET))
    assert_matches_oracle(device_assembly(pkg, part, d, "newton", None, (gd, gv)), oracle_assembly(pkg, name, "newton"), part)


def test_valence_65_is_refused(pkg):
    m, d, part = case(pkg, "wheel65")
    with pytest.raises(Exception, match="a vertex has 65 incident cells"):
        pkg.DeviceProblem(part, 0)


def test_fallback_mixed_orientation_to_variant4(pkg):
    """Half of the cells (seeded) listed clockwise: the fan scheme refuses, the default assembly is variant 4's, and it matches
    the oracle on the original mesh."""
    m, d, part = case(pkg, "delaunay3000")
    fl = mg.flipped(part, np.random.default_rng(4).random(part.n_cells) < 0.5)
    out = all_variants(pkg, fl, d)
    assert "valence <= 32" in out[5]
    assert same(out["default"], out[4]) and not same(out["default"], out[0])
    gd, gv = d.dirichlet_values(mg.CALLS, dict(time_factor=1.0, **mg.INLET))
    for mode in ("newton", "stokes"):
        assert_matches_oracle(device_assembly(pkg, fl, d, mode, None, (gd, gv)), oracle_assembly(pkg, "delaunay3000", mode), part)


@pytest.mark.parametrize("variant", [0, 4, 5])
def test_all_cells_clockwise(pkg, variant):
    """Every cell listed clockwise is again an oriented triangulation: the fan scheme serves it (fans run the other way round),
    and every variant matches the oracle on the original mesh."""
    m, d, part = case(pkg, "delaunay3000")
    fl = mg.flipped(part, np.arange(part.n_cells))
    if variant == 5:
        out = all_variants(pkg, fl, d)
        assert same(out["default"], out[5])
    gd, gv = d.dirichlet_values(mg.CALLS, dict(time_factor=1.0, **mg.INLET))
    for mode in ("newton", "stokes"):
        assert_matches_oracle(device_assembly(pkg, fl, d, mode, variant, (gd, gv)), oracle_assembly(pkg, "delaunay3000", mode), part)
