"""The C++ host shim (navier-stokes-dealii_b200/host): the reference's own src/main.cpp must compile and
link against it UNCHANGED (SURVEY §8b), and the app must fail loudly without a GPU."""
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, mesh_path

HOST = os.path.join(ROOT, "navier-stokes-dealii_b200", "host")
# the reference's src/main.cpp (tests/golden/README.md); NS_REFERENCE_MAIN points at the original file instead
REF_MAIN = os.environ.get("NS_REFERENCE_MAIN", mesh_path("reference_main.cpp"))


def test_reference_main_compiles_and_links_unchanged(tmp_path):
    # `#include "NavierStokesSolver.hpp"` resolves next to main.cpp first, so build it from a scratch
    # directory (outside the repo) the way a maintainer would after dropping the shim header into src/
    import shutil
    main_cpp = tmp_path / "main.cpp"
    shutil.copyfile(REF_MAIN, main_cpp)
    exe = tmp_path / "proj"
    cmd = ["g++", "-std=c++17", "-O1", f"-I{HOST}", f"-I{ROOT}/include", str(main_cpp),
           os.path.join(HOST, "NavierStokesSolver.cpp"), f"-L{ROOT}/navier-stokes-dealii_b200", "-lnst", "-lnsg",
           f"-Wl,-rpath,{ROOT}/navier-stokes-dealii_b200", "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert exe.exists()


def test_app_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    env = dict(os.environ, NS_MESH=mesh_path("square_h0.1.msh"))
    r = subprocess.run([os.path.join(HOST, "ns_app")], capture_output=True, text=True, env=env)
    assert r.returncode == 1 and "no CUDA device" in r.stderr


@pytest.mark.gpu
def test_app_matches_python_driver(pkg):
    """ns_app (C++ shim) and the Python mirror drive the same C-ABI: identical Newton/GMRES record."""
    env = dict(os.environ, NS_MESH=mesh_path("cylinder_cmy.msh"), NS_T="0.05")
    r = subprocess.run([os.path.join(HOST, "ns_app"), "--history"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    recs = [json.loads(line) for line in r.stdout.splitlines() if line.startswith("{")]
    assert "Number of elements = 6448" in r.stdout and "total    = 29646" in r.stdout
    s = pkg.NavierStokesSolver(2, 1, 0.05, 0.05, pkg.Parameters(mesh_path=mesh_path("cylinder_cmy.msh")), verbose=False)
    s.setup()
    s.solve()
    assert len(recs) == len(s.history) >= 2
    for a, (step, it, res, its) in zip(recs, s.history):
        assert (a["time_step"], a["newton"]) == (step, it)
        assert a["gmres"] == (-1 if its is None else its)
        assert a["residual"] == res          # same library, same device: bit-identical


@pytest.mark.gpu
def test_app_writes_output_files(tmp_path):
    """N2: output() keeps the reference's one-file-per-step contract (cpp:681-728) as XDMF + raw binary heavy data and as legacy VTK."""
    env = dict(os.environ, NS_MESH=mesh_path("square_h0.1.msh"), NS_T="0.1", NS_NEUMANN_ID="1", NS_INLET_ID="0",
               NS_WALL_IDS="2,3", NS_OUTPUT_DIR=str(tmp_path))
    r = subprocess.run([os.path.join(HOST, "ns_app")], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    files = sorted(os.listdir(tmp_path))
    assert [f for f in files if f.endswith(".vtk")] == ["output-0000.rank0.vtk", "output-0001.rank0.vtk", "output-0002.rank0.vtk"]
    assert [f for f in files if f.endswith(".xdmf")] == ["output-0000.xdmf", "output-0001.xdmf", "output-0002.xdmf"]
    txt = open(os.path.join(tmp_path, "output-0002.rank0.vtk")).read()
    assert "CELLS 200 800" in txt and "VECTORS velocity double" in txt and "SCALARS pressure double 1" in txt
    assert "SCALARS partitioning int 1" in txt and "nan" not in txt
    # the XDMF + raw-binary files of the C++ host are the ones the Python mirror reads back
    import importlib
    import numpy as np
    xout = importlib.import_module("navier-stokes-dealii_b200.output")
    t, grids = xout.read_back(str(tmp_path), "output-0002.xdmf")
    r = grids["rank0"]
    assert abs(t - 0.1) < 1e-12 and r["cells"].shape == (200, 3) and r["points"].shape == (600, 2)
    assert np.isfinite(r["velocity"]).all() and np.abs(r["velocity"][:, :2]).max() > 0 and not r["velocity"][:, 2].any()
    assert (r["partitioning"] == 0).all()
