"""Collective point evaluation on P GPUs: run under  python -m torch.distributed.run --nproc-per-node P scripts/points_check.py
Every rank owns one RCB partition of cylinder_cmy.msh, all ranks evaluate the same points collectively (NCCL), and each
rank compares its result with a 1-rank context on its own GPU: cell ids, values and gradients must be bitwise equal.  A
short solver run with probes checks that every rank records the same probe history.  Each rank writes
$POINTS_RESULT_DIR/rank<r>.json."""
import importlib
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
pkg = importlib.import_module("navier-stokes-dealii_b200")
from conftest import analytic_state, mesh_path  # noqa: E402


def fresh_unique_id(rank):
    """An NCCL unique id serves one communicator: every communicator gets its own, made on rank 0 and broadcast."""
    uid = [pkg.DeviceProblem.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    return uid[0]


def main():
    # a stuck collective must not hang the GPU box: dump every thread's Python stack and exit
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("POINTS_WATCHDOG_S", "240")), exit=True)
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    m = pkg.Mesh.read_msh(mesh_path("cylinder_cmy.msh"))
    rng = np.random.default_rng(7)
    xy, ev = m.xy, m.edge_vertices
    lo, hi = xy.min(0), xy.max(0)
    pts = np.concatenate([lo + (hi - lo) * rng.random((4000, 2)), xy, 0.5 * (xy[ev[:, 0]] + xy[ev[:, 1]]),
                          [[-0.5, -2.31253069e-09], [0.5, 2.31253069e-09], [1e3, 0.0], [np.nan, 0.0]]])

    d1 = pkg.Dofs(m)
    p1 = pkg.Part(d1, 0, patterns=False)
    one = pkg.DeviceProblem(p1, local)
    one.set_solution(analytic_state(d1)[np.asarray(p1.l2g[: p1.n_own])])
    ref = one.evaluate(pts, gradients=True)
    one.close()

    cp = m.partition_rcb(world)
    d = pkg.Dofs(m, world, cp)
    part = pkg.Part(d, rank, patterns=False)
    dev = pkg.DeviceProblem(part, local)
    dev.comm_init(rank, world, fresh_unique_id(rank))
    dev.set_solution(analytic_state(d)[np.asarray(part.l2g[: part.n_own])])   # owned entries; the halo exchange fills the ghosts
    vals, grads, cells = dev.evaluate(pts, gradients=True)                        # collective: comm_init was called
    res = dict(rank=rank, world=world, n_points=len(pts), found=int((cells >= 0).sum()),
               cells_equal=bool(np.array_equal(cells, ref[2])),
               values_bitwise=bool(np.array_equal(vals.view(np.uint64), ref[0].view(np.uint64))),
               grads_bitwise=bool(np.array_equal(np.ascontiguousarray(grads).view(np.uint64),
                                                 np.ascontiguousarray(ref[1]).view(np.uint64))))
    dev.close()

    # solver level: two time steps with probes on every rank, gathered and compared
    prm = pkg.Parameters(mesh_path=mesh_path("square_h0.1.msh"), nu=0.05, H=1.0, inlet_time_mode="constant", neumann_id=1,
                         inlet_id=0, wall_ids=(2, 3), clear_inlet_before_walls=True, preconditioner="identity", p_out=0.0,
                         increment_bc="consistent", newton_max_iters=3, probe_points=((0.5, 0.5), (0.25, 0.75), (0.8, 0.1)))
    s = pkg.NavierStokesSolver(2, 1, 0.1, 0.05, prm, device=local, rank=rank, world_size=world,
                               comm_unique_id=fresh_unique_id(rank), verbose=False)
    s.setup()
    s.solve()
    hist = [(t, v.tolist()) for t, v in s.probe_history]
    every = [None] * world
    dist.all_gather_object(every, hist)
    res["probe_history_equal"] = len(hist) == 2 and all(h == hist for h in every) and not np.isnan(np.array(hist[-1][1])).any()
    s.dev.close()

    out_dir = os.environ.get("POINTS_RESULT_DIR", "points_check_out")
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, f"rank{rank}.json"), "w") as f:
        json.dump(res, f)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("POINTS_CHECK", "PASS" if all(v for k, v in res.items() if k.endswith(("equal", "bitwise"))) else "FAIL", flush=True)


if __name__ == "__main__":
    main()
