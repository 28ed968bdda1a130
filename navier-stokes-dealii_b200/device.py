"""Thin object wrapper over the device C-ABI (include/nsg.h). One instance = one GPU = one rank."""
import ctypes as C

import numpy as np

from ._lib import NsgParams, nsg, nsg_check

PRECOND_IDENTITY, PRECOND_BLOCK_DIAGONAL, PRECOND_BLOCK_TRIANGULAR = 0, 1, 2


class DeviceProblem:
    def __init__(self, part, device=0, stream=None):
        """part: topology.Part. Uploads the fixed CSR and the mesh tables once."""
        L = nsg()
        self._L = L
        h = C.c_void_p()
        nsg_check(L.nsg_create(int(device), C.byref(h)))
        self._h = h
        self.part = part
        self.n_own = part.n_own
        self.nnz = part.nnz_jac
        self.pm_nnz = part.nnz_pm
        if stream is not None:
            nsg_check(L.nsg_set_stream(h, C.c_void_p(int(stream))))
        if getattr(part, "has_patterns", True):
            nsg_check(L.nsg_set_pattern(h, part.n_own_u, part.n_own_p, part.n_ghost_u, part.n_ghost_p, part.jac_rowptr,
                                        _nz(part.jac_col), part.pm_rowptr, _nz(part.pm_col)))
        else:   # Part(..., patterns=False): the device builds the two sparsity patterns from the cell -> dof table (N4)
            nsg_check(L.nsg_set_pattern_from_cells(h, part.n_own_u, part.n_own_p, part.n_ghost_u, part.n_ghost_p, part.n_cells,
                                                   _nz(part.cell_dofs)))
            a, b = C.c_int64(), C.c_int64()
            nsg_check(L.nsg_get_pattern_sizes(h, C.byref(a), C.byref(b)))
            self.nnz, self.pm_nnz = a.value, b.value
        nsg_check(L.nsg_set_mesh(h, part.n_cells, part.n_vertices, part.xy, part.cell_vertices, part.cell_dofs,
                                 len(part.bface_cell), _nz(part.bface_cell), _nz(part.bface_face), _nz(part.bface_tag)))
        self.params = NsgParams()
        L.nsg_params_default(C.byref(self.params))

    # -- multi-GPU plumbing -------------------------------------------------------------------
    @staticmethod
    def comm_unique_id():
        buf = C.create_string_buffer(128)
        nsg_check(nsg().nsg_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, rank, n_ranks, unique_id):
        nsg_check(self._L.nsg_comm_init(self._h, int(rank), int(n_ranks), C.create_string_buffer(unique_id, 128)))
        self._comm = True
        p = self.part
        nsg_check(self._L.nsg_set_halo(self._h, p.n_neighbors, _nz(p.neighbors), p.send_ptr, _nz(p.send_idx), p.recv_ptr,
                                       _nz(p.recv_idx)))

    def comm_ipc_handle(self):
        buf = C.create_string_buffer(64)
        nsg_check(self._L.nsg_comm_ipc_handle(self._h, buf))
        return buf.raw

    def comm_set_peers(self, handles):
        """handles: list of the 64-byte IPC handles of all ranks in rank order (fused NVLink all-reduce)."""
        blob = b"".join(handles)
        nsg_check(self._L.nsg_comm_set_peers(self._h, C.create_string_buffer(blob, len(blob))))

    def enable_peer_allreduce(self, dist):
        """All ranks: exchange the mailbox handles over torch.distributed and switch the Krylov inner products to
        the all-reduce fused into the reduction kernels (NVLink peer memory).  NSG_NO_PEER_AR=1 keeps NCCL."""
        import os
        if os.environ.get("NSG_NO_PEER_AR", "0") == "1" or dist.get_world_size() <= 1:
            return False
        # a rank that cannot export or map a mailbox (no peer access between the devices) must not leave the others
        # spinning on it: the decision to switch is taken collectively, otherwise everybody stays on NCCL
        world = dist.get_world_size()
        try:
            mine, err = self.comm_ipc_handle(), None
        except Exception as e:  # noqa: BLE001
            mine, err = b"\0" * 64, str(e)
        handles = [None] * world
        dist.all_gather_object(handles, (mine, err))
        if all(e is None for _, e in handles):
            try:
                self.comm_set_peers([h for h, _ in handles])
            except Exception as e:  # noqa: BLE001
                err = str(e)
        ok = [None] * world
        dist.all_gather_object(ok, err is None and all(e is None for _, e in handles))
        if not all(ok):
            self._L.nsg_comm_release_peers(self._h)   # closes whatever was mapped; reductions stay on NCCL
            dist.barrier()
            return False
        dist.barrier()
        self._peer_dist = dist   # close() releases the peer mappings collectively before freeing the mailbox
        return True

    # -- parameters -----------------------------------------------------------------------------
    def set_params(self, **kw):
        for k, v in kw.items():
            if k == "forcing":
                self.params.forcing[0], self.params.forcing[1] = v
            else:
                setattr(self.params, k, v)
        nsg_check(self._L.nsg_set_params(self._h, C.byref(self.params)))

    # -- hot path ---------------------------------------------------------------------------------
    def assemble(self):
        nsg_check(self._L.nsg_assemble(self._h))

    def apply_dirichlet(self, dofs, values, into_solution=False):
        dofs = np.ascontiguousarray(dofs, np.int32)
        values = np.ascontiguousarray(values, np.float64)
        nsg_check(self._L.nsg_apply_dirichlet(self._h, len(dofs), _nz(dofs), _nz(values, np.float64),
                                              1 if into_solution else 0))

    def residual_norm(self):
        out = C.c_double()
        nsg_check(self._L.nsg_residual_norm(self._h, C.byref(out)))
        return out.value

    def solve(self, precond=PRECOND_IDENTITY, rel_tol=1e-2, max_it=100000, n_tmp=30, target=0, check=True):
        its, res = C.c_int32(), C.c_double()
        rc = self._L.nsg_solve(self._h, precond, rel_tol, max_it, n_tmp, target, C.byref(its), C.byref(res))
        if check:
            nsg_check(rc)
        return its.value, res.value, rc

    def gmres_history(self):
        n = self._L.nsg_gmres_history(self._h, None, 0)
        out = np.zeros(max(n, 1), np.float64)
        self._L.nsg_gmres_history(self._h, out, n)
        return out[:n]

    def last_solve_info(self):
        """Which path the last solve() took: dict(fused, graph_replays, spmv_variant, orthogonalization)."""
        out = np.zeros(4, np.int32)
        nsg_check(self._L.nsg_last_solve_info(self._h, out))
        return {"fused": bool(out[0]), "graph_replays": int(out[1]), "spmv_variant": int(out[2]), "orthogonalization": int(out[3])}

    def last_inner_iterations(self):
        """Inner CG / GMRES iterations (= ILU(0) applies) of the block preconditioner during the last solve()."""
        return int(self._L.nsg_last_inner_iterations(self._h))

    def get_pattern(self):
        """(jac_rowptr, jac_col, pm_rowptr, pm_col) as the device holds them."""
        rp, prp = np.zeros(self.n_own + 1, np.int64), np.zeros(self.n_own + 1, np.int64)
        col, pcol = np.zeros(max(self.nnz, 1), np.int32), np.zeros(max(self.pm_nnz, 1), np.int32)
        nsg_check(self._L.nsg_get_pattern(self._h, rp, col, prp, pcol))
        return rp, col[: self.nnz], prp, pcol[: self.pm_nnz]

    def update_solution(self):
        nsg_check(self._L.nsg_update_solution(self._h))

    def push_time_level(self):
        nsg_check(self._L.nsg_push_time_level(self._h))

    # -- host <-> device ---------------------------------------------------------------------------
    def _set(self, fn, v):
        v = np.ascontiguousarray(v, np.float64)
        assert v.shape == (self.n_own,), f"expected {self.n_own} owned entries, got {v.shape}"
        nsg_check(fn(self._h, v))

    def _get(self, fn, n, out=None):
        if out is None:
            out = np.zeros(max(n, 1), np.float64)
        nsg_check(fn(self._h, out))
        return out[:n]

    def set_solution(self, v):
        self._set(self._L.nsg_set_solution, v)

    def set_solution_old(self, v):
        self._set(self._L.nsg_set_solution_old, v)

    def set_delta(self, v):
        self._set(self._L.nsg_set_delta, v)

    def get_solution(self):
        return self._get(self._L.nsg_get_solution, self.n_own)

    def get_solution_ghosted(self):
        """Owned entries followed by the ghost layer (the vector `solution` of the reference, hpp:791)."""
        return self._get(self._L.nsg_get_solution_ghosted, self.part.n_loc)

    def get_delta(self, out=None):
        """out: optional preallocated (e.g. page-locked) float64 array of n_own entries."""
        return self._get(self._L.nsg_get_delta, self.n_own, out)

    def get_residual(self):
        return self._get(self._L.nsg_get_residual, self.n_own)

    def get_matrix_values(self):
        return self._get(self._L.nsg_get_matrix_values, self.nnz)

    def get_pm_values(self):
        return self._get(self._L.nsg_get_pm_values, self.pm_nnz)

    def set_solution_ghosted(self, v):
        """Owned entries followed by the ghost layer, written as given (no exchange): the inverse of get_solution_ghosted."""
        v = np.ascontiguousarray(v, np.float64)
        if v.shape != (self.part.n_loc,):
            raise ValueError(f"expected {self.part.n_loc} owned + ghost entries, got {v.shape}")
        nsg_check(self._L.nsg_set_solution_ghosted(self._h, v))

    def boundary_force(self, boundary_id):
        """(drag, lift) on the body bounded by the faces with this boundary id (N3)."""
        out = np.zeros(2)
        nsg_check(self._L.nsg_boundary_force(self._h, int(boundary_id), out))
        return out

    def evaluate(self, points, gradients=False, collective=None):
        """u_x, u_y, p of the current solution at points (n, 2): returns values (n, 3), then grads (n, 2, 3) with
        grads[i, d, k] = d(value k)/dx_d if gradients, then cells (n,), the global id of the cell used (-1 and NaN values
        where no cell contains the point). collective=None: collective exactly when comm_init was called; then every rank
        passes the same points and gets the same results."""
        pts = np.ascontiguousarray(points, np.float64)
        if pts.ndim != 2 or pts.shape[1] != 2:
            raise ValueError(f"points must have shape (n, 2), got {pts.shape}")
        if not getattr(self, "_ownership_set", False):   # first use: global cell ids and ownership of the partition
            nsg_check(self._L.nsg_set_cell_ownership(self._h, _nz(self.part.cell_ids), _nz(self.part.cell_owned, np.uint8)))
            self._ownership_set = True
        if collective is None:
            collective = getattr(self, "_comm", False)
        n = len(pts)
        vals = np.empty((max(n, 1), 3), np.float64)
        grads = np.empty((max(n, 1), 3, 2), np.float64) if gradients else None
        cells = np.empty(max(n, 1), np.int64)
        nsg_check(self._L.nsg_eval_points(self._h, n, _nz(pts.reshape(-1), np.float64), 1 if collective else 0, vals.reshape(-1),
                                          None if grads is None else grads.reshape(-1), cells))
        return (vals[:n],) + ((grads[:n].transpose(0, 2, 1),) if gradients else ()) + (cells[:n],)

    def points_index_info(self):
        """The spatial index of evaluate() (built by its first call)."""
        o = np.zeros(8)
        nsg_check(self._L.nsg_points_index_info(self._h, o))
        return {"bins_x": int(o[0]), "bins_y": int(o[1]), "bin_side": o[2], "entries": int(o[3]), "nonempty_bins": int(o[4]),
                "max_bin": int(o[5]), "bytes": int(o[6]), "build_ms": o[7]}

    def spmv(self, x):
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros(self.n_own, np.float64)
        nsg_check(self._L.nsg_spmv(self._h, x, y))
        return y

    def precond_apply(self, precond, x):
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros(self.n_own, np.float64)
        nsg_check(self._L.nsg_precond_apply(self._h, precond, x, y))
        return y

    def ilu_apply(self, which, x):
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros(len(x), np.float64)
        nsg_check(self._L.nsg_ilu_apply(self._h, which, x, y))
        return y

    def time_kernel(self, what, reps):
        ms = C.c_double()
        nsg_check(self._L.nsg_time_kernel(self._h, what, reps, C.byref(ms)))
        return ms.value

    def set_tuning(self, key, value):
        nsg_check(self._L.nsg_set_tuning(self._h, int(key), int(value)))

    def counters(self):
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        nsg_check(self._L.nsg_get_counters(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return {"launches": a.value, "h2d_bytes": b.value, "d2h_bytes": c.value}

    def phase_ms(self):
        out = (C.c_double * 3)()
        nsg_check(self._L.nsg_get_phase_ms(self._h, out))
        return {"assemble": out[0], "dirichlet": out[1], "solve": out[2]}

    def close(self):
        """Collective when the fused all-reduce is on (every rank must call it): the peers' mailbox mappings are
        closed on every rank, then a barrier, and only then is any mailbox freed (CUDA IPC rule)."""
        if getattr(self, "_h", None):
            dist = getattr(self, "_peer_dist", None)
            if dist is not None:
                self._L.nsg_comm_release_peers(self._h)
                self._peer_dist = None
                try:
                    dist.barrier()
                except Exception:
                    pass
            self._L.nsg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self._peer_dist = None   # no collectives from a finaliser
            self.close()
        except Exception:
            pass


def _nz(a, dtype=np.int32):
    """ctypes ndpointer needs a real buffer even for empty arrays."""
    a = np.ascontiguousarray(a, dtype)
    return a if a.size else np.zeros(1, dtype)
