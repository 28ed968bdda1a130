"""-m gpu: `bench.py --dump-outputs` on a small workload writes what its timed step computed - checked against the CPU oracle
run on the same inputs, entry by entry at the global (row, column) keys of the dump."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import ROOT
from oracle.oracle import Oracle

pytestmark = pytest.mark.gpu

FILES = ["gmres_residual_history", "jacobian_cols", "jacobian_rows", "jacobian_values", "newton_increment",
         "pressure_mass_cols", "pressure_mass_rows", "pressure_mass_values", "residual", "sample_dofs", "step_scalars"]


def test_bench_dump_outputs_match_the_oracle(pkg, tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--mesh", "cmy", "--levels", "0", "--steps", "1",
           "--warmup", "0", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(got) == FILES and all(a.dtype == np.float64 for a in got.values())

    # the same inputs on the CPU oracle: bench's own problem set-up and parameters
    m, d, part, (ld, lv), neumann, sol = bench.build_problem(pkg, "cmy", 0, 1, 0)
    o = Oracle(part)
    o.set_params(neumann_id=neumann, nu=0.001, deltat=0.05)
    o.set_solution(sol)
    o.set_solution_old(0.9 * sol)
    o.set_delta(np.zeros(d.n))
    o.assemble()
    o.apply_dirichlet(ld, lv)
    its, res, rc = o.solve(0, 1e-2, 56, 30, 0)
    g2l = np.empty(d.n, np.int64)
    g2l[part.l2g] = np.arange(d.n)

    # vectors: every DoF (n <= DUMP_SAMPLE)
    assert d.n <= bench.DUMP_SAMPLE and np.array_equal(got["sample_dofs"], np.arange(d.n))
    R = o.get_residual()[g2l]
    assert np.abs(got["residual"] - R).max() <= 1e-12 * np.abs(R).max()
    delta = o.get_delta()[g2l]
    assert np.abs(got["newton_increment"] - delta).max() <= 1e-8 * np.abs(delta).max()
    norm, steps, final = got["step_scalars"]
    assert abs(norm - o.residual_norm()) <= 1e-12 * o.residual_norm()
    assert abs(np.linalg.norm(got["residual"]) - norm) <= 1e-12 * norm
    h = o.gmres_history()
    assert steps == its == len(got["gmres_residual_history"]) and abs(final - res) <= 1e-8 * res
    assert np.abs(got["gmres_residual_history"] / h - 1).max() <= 1e-8

    # matrices: every stored entry of the sampled rows (n > DUMP_ROWS), keyed by global (row, column)
    rows = bench._sample(d.n, bench.DUMP_ROWS, 1)
    assert len(rows) < d.n
    for name, values, rp, col in (("jacobian", o.get_matrix_values(), part.jac_rowptr, part.jac_col),
                                  ("pressure_mass", o.get_pm_values(), part.pm_rowptr, part.pm_col)):
        A = sp.csr_matrix((values, col, rp), shape=(d.n, d.n))
        i, j = g2l[got[f"{name}_rows"].astype(np.int64)], g2l[got[f"{name}_cols"].astype(np.int64)]
        v = got[f"{name}_values"]
        assert len(v) == np.diff(rp)[g2l[rows]].sum() > 0, name
        assert np.isin(part.l2g[i], rows).all() and (np.diff(got[f"{name}_rows"]) >= 0).all(), name
        want = np.asarray(A[i, j]).ravel()
        scale = abs(A).max(axis=1).toarray().ravel()[i]     # entries are sums of cancelling cell contributions
        scale[scale == 0] = 1.0
        assert (np.abs(v - want) <= 1e-12 * scale).all(), name
