/* nsg.h — device C-ABI (libnsg.so): the per-Newton-step hot path of
 * NavierStokesSolver on one B200 per process (CUDA, sm_100a, fp64).
 *
 * This is the boundary BASELINE.json:north_star names: the Trilinos objects on the
 * path (TrilinosWrappers::BlockSparseMatrix jacobian_matrix / pressure_mass and the
 * MPI::BlockVector residual_vector / delta_owned / solution_owned / solution /
 * solution_old, /root/reference src/NavierStokesSolver.hpp:765-794) are replaced by a
 * fixed device CSR and device vectors owned by an opaque context; the class methods
 * that touch them call the entry points below.  Each entry point cites the reference
 * lines it replaces (paths relative to /root/reference).
 *
 * Conventions: extern "C", plain pointers and sizes, no exceptions across the
 * boundary.  Every function returns NSG_OK or a negative NSG_ERR_* code;
 * nsg_last_error() gives the text for the calling thread.  All host buffers are
 * caller-owned and may be freed when the call returns.  One context drives one GPU;
 * calls on a context are not re-entrant; all device work is ordered on the context's
 * stream.  There is NO CPU fallback: without a CUDA device nsg_create fails.
 *
 * Local numbering of a context (one rank of P; for P = 1 "local" = "global"):
 *   [ owned u | owned p | ghost u | ghost p ],  rows of every matrix = owned DoFs,
 *   columns = local ids ascending.  include/nst.h (nst_part_*) produces all inputs.
 */
#ifndef NSG_H
#define NSG_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define NSG_OK 0
#define NSG_ERR_CUDA (-1)
#define NSG_ERR_ARG (-2)
#define NSG_ERR_NO_CONVERGENCE (-3)       /* SolverControl::NoConvergence of the outer GMRES */
#define NSG_ERR_INNER_NO_CONVERGENCE (-4) /* ... of an inner CG/GMRES of a block preconditioner */
#define NSG_ERR_STATE (-5)                /* call order violated (e.g. assemble before set_mesh) */
#define NSG_ERR_NCCL (-6)

#define NSG_PRECOND_IDENTITY 0          /* hpp:504-517, the one solve_system uses (cpp:570) */
#define NSG_PRECOND_BLOCK_DIAGONAL 1    /* hpp:520-572 */
#define NSG_PRECOND_BLOCK_TRIANGULAR 2  /* hpp:575-639 */

typedef struct nsg_ctx nsg_ctx;

const char *nsg_last_error(void);

/* device = CUDA ordinal this context owns. */
int nsg_create(int device, nsg_ctx **out);
void nsg_destroy(nsg_ctx *ctx);

/* Run all device work of this context on an existing CUDA stream (cudaStream_t passed as
 * void*), e.g. torch's current stream so that torch.cuda.Event brackets it; NULL = own stream. */
int nsg_set_stream(nsg_ctx *ctx, void *cuda_stream);

/* jacobian_matrix.reinit(sparsity), pressure_mass.reinit(...), vector reinit x5
 * (cpp:161-174): uploads the FIXED patterns once and allocates all device vectors.
 * jac_rowptr/pm_rowptr have n_own_u+n_own_p+1 entries (int64: nnz may pass 2^31). */
int nsg_set_pattern(nsg_ctx *ctx, int64_t n_own_u, int64_t n_own_p, int64_t n_ghost_u, int64_t n_ghost_p,
                    const int64_t *jac_rowptr, const int32_t *jac_col, const int64_t *pm_rowptr,
                    const int32_t *pm_col);

/* SURVEY 8f N4 - the same two patterns (DoFTools::make_sparsity_pattern, cpp:107-110 full coupling; cpp:143-158 p-p only)
 * built ON THE DEVICE from the cell -> dof table instead of uploaded: bit-identical to the patterns of nst_part_build
 * (tests/test_gpu_parity.py::test_device_pattern_is_bit_identical), without the host construction, the host copies and the
 * upload of ~10 GB of column indices at 85 M DoFs. cell_dofs[15*n_cells] as for nsg_set_mesh. Use INSTEAD of
 * nsg_set_pattern; nsg_get_pattern_sizes / nsg_get_pattern read the result back (sizes; rowptr n_own+1, col nnz). */
int nsg_set_pattern_from_cells(nsg_ctx *ctx, int64_t n_own_u, int64_t n_own_p, int64_t n_ghost_u, int64_t n_ghost_p,
                               int64_t n_cells, const int32_t *cell_dofs);
int nsg_get_pattern_sizes(nsg_ctx *ctx, int64_t *nnz_jac, int64_t *nnz_pm);
int nsg_get_pattern(nsg_ctx *ctx, int64_t *jac_rowptr, int32_t *jac_col, int64_t *pm_rowptr, int32_t *pm_col);

/* What the cell loop reads through deal.II (cell->vertex, get_dof_indices, boundary_id;
 * cpp:218-343): vertex coordinates xy[2*n_vertices], cell_vertices[3*n_cells],
 * cell_dofs[15*n_cells] (local ids, FESystem order: 3v+{0,1} u, 3v+2 p, 9+2l+{0,1} u),
 * and the boundary faces (cell, local face 0..2, boundary id). Call after nsg_set_pattern. */
int nsg_set_mesh(nsg_ctx *ctx, int64_t n_cells, int64_t n_vertices, const double *xy,
                 const int32_t *cell_vertices, const int32_t *cell_dofs, int64_t n_bfaces,
                 const int32_t *bface_cell, const int32_t *bface_face, const int32_t *bface_tag);

/* Ghost import plan (Epetra Import behind `solution = solution_owned`, cpp:587,618, and
 * behind every vmult): see nst_part_neighbors, nst_part_send_idx, nst_part_recv_idx. Only needed for P > 1. */
int nsg_set_halo(nsg_ctx *ctx, int32_t n_neighbors, const int32_t *neighbors, const int64_t *send_ptr,
                 const int32_t *send_idx, const int64_t *recv_ptr, const int32_t *recv_idx);

/* NCCL communicator over NVLink (replaces MPI_COMM_WORLD, hpp:646-653). unique_id is the
 * 128-byte ncclUniqueId created on rank 0 by nsg_comm_unique_id and broadcast by the host. */
int nsg_comm_unique_id(void *out128);
int nsg_comm_init(nsg_ctx *ctx, int rank, int n_ranks, const void *unique_id128);

/* Optional, after nsg_comm_init on every rank: fuse the scalar all-reduces of the Krylov inner products
 * (MPI_Allreduce behind every dot/norm of SolverGMRES, SURVEY 2.2) into the reduction kernels as a one-shot
 * exchange through NVLink peer memory. Each rank exports the CUDA-IPC handle of its mailbox (64 bytes), the
 * host all-gathers them in rank order, nsg_comm_set_peers maps them. Without it NCCL does the all-reduce. */
int nsg_comm_ipc_handle(nsg_ctx *ctx, void *out64);
int nsg_comm_set_peers(nsg_ctx *ctx, const void *handles /* n_ranks x 64 bytes, rank order */);
/* Unmap the peers' mailboxes and go back to NCCL all-reduces. Every rank must call this and then synchronise with the
 * others (barrier) BEFORE any rank destroys its context: CUDA IPC requires importers to close a mapping before the
 * exporter frees the memory. */
int nsg_comm_release_peers(nsg_ctx *ctx);

/* The compile-time constants of the reference as run-time parameters; defaults are the
 * reference's values (hpp:703-709 nu,rho,p_out; main.cpp:13 deltat; hpp:438 g=0; cpp:320 id 10). */
typedef struct {
  double nu, rho, p_out;
  double deltat;       /* used when use_mass != 0 */
  double forcing[2];   /* f = (0,-g) */
  int32_t neumann_id;  /* boundary id of the Neumann (p_out) faces */
  int32_t use_mass;    /* 1 = implicit Euler terms (cpp:249-251, 288-290); 0 = steady */
  int32_t stokes;      /* 1 = assemble_stokes_system (cpp:380-531) into the same objects */
  int32_t dirichlet_diag; /* diagonal of a constrained row after nsg_apply_dirichlet (cpp:375-376):
                           0 (default) = TrilinosWrappers rule: ALWAYS replaced by d = |first non-zero diagonal entry of
                           the block's locally owned rows|, rhs_i = g_i d (MatrixTools::apply_boundary_values for Trilinos
                           matrices: clear_rows(rows, d)); 1 = deal.II's native-SparseMatrix rule: a non-zero diagonal
                           is kept (d only where it is zero), rhs_i = g_i J_ii */
} nsg_params;
void nsg_params_default(nsg_params *p);
int nsg_set_params(nsg_ctx *ctx, const nsg_params *p);

/* assemble_system up to and including compress(add) (cpp:203-347): J = 0, R = 0, Mp = 0, the cell
 * loop with the Neumann faces, and the scatter into the fixed CSR — one call, no per-cell host
 * traffic. Reads `solution` and `solution_old` (ghosts must be current: nsg_set_solution,
 * nsg_update_solution and nsg_push_time_level keep them so). The pressure rows of J and Mp depend
 * on the geometry and nu only: they are integrated by the first call and again only after nu,
 * the assembly variant or a Dirichlet constraint on a pressure row changed them; R_p = 0 is
 * written by every call. */
int nsg_assemble(nsg_ctx *ctx);

/* MatrixTools::apply_boundary_values(bv, jacobian_matrix, delta_owned, residual_vector, false)
 * (cpp:375-376) for the (dof, value) list the host evaluated with interpolate_boundary_values
 * (cpp:351-373); dofs are LOCAL owned ids. into_solution != 0 is the Stokes call (cpp:529): the
 * reference passes the GHOSTED `solution` there, which solve_stokes_system neither reads (it iterates
 * on solution_owned) nor keeps (it is overwritten by the ghost import, cpp:556) - so only the matrix
 * rows and the right-hand side are modified and no vector entry is written. */
int nsg_apply_dirichlet(nsg_ctx *ctx, int64_t n, const int32_t *dofs, const double *values, int32_t into_solution);

/* residual_vector.l2_norm() (cpp:602,566): global over all ranks; synchronises. */
int nsg_residual_norm(nsg_ctx *ctx, double *out);

/* solve_system (cpp:561-588): SolverControl(max_it, rel_tol*||R||), deal.II SolverGMRES with
 * n_tmp_vectors temporaries (30 -> restart every 28 steps), left preconditioning, x0 = current
 * delta (target 0) or solution (target 1: solve_stokes_system, cpp:533-559), then the ghost
 * import. its_out = SolverControl::last_step(), res_out = last residual estimate. */
int nsg_solve(nsg_ctx *ctx, int32_t precond, double rel_tol, int32_t max_it, int32_t n_tmp_vectors,
              int32_t target, int32_t *its_out, double *res_out);
/* residual estimate after every GMRES step of the last nsg_solve (returns how many exist). */
int64_t nsg_gmres_history(nsg_ctx *ctx, double *out, int64_t cap);
/* Which code path the last nsg_solve took (so that a test can assert that the knob it set was the one exercised):
 * out4[0] = 1 the whole solve ran as the ONE cooperative kernel (tuning key 5), 0 the multi-kernel solver;
 * out4[1] = number of CUDA-graph replays of restart-cycle segments (tuning key 2; 0 = plain launches);
 * out4[2] = SpMV kernel variant used by the operator (tuning key 0; -1 for the cooperative kernel, which has its own);
 * out4[3] = Gram-Schmidt variant (tuning key 3). */
int nsg_last_solve_info(nsg_ctx *ctx, int32_t *out4);
/* Iterations the inner CG / GMRES solvers of a block preconditioner (hpp:541-551, 598-612) took during the last nsg_solve, summed
 * over its applications (each inner iteration is one ILU(0) apply); 0 for the identity. Returns the count. */
int64_t nsg_last_inner_iterations(nsg_ctx *ctx);

/* solution_owned += delta_owned; solution = solution_owned (cpp:616-618). */
int nsg_update_solution(nsg_ctx *ctx);
/* solution_old = solution (cpp:666). */
int nsg_push_time_level(nsg_ctx *ctx);

/* Host <-> device copies of the OWNED entries (n_own_u + n_own_p doubles, local order).
 * set_* also refresh the ghosts. VectorTools::interpolate + ghost import (cpp:650-651), and
 * what output() reads (cpp:697-700). */
int nsg_set_solution(nsg_ctx *ctx, const double *host);
int nsg_set_solution_old(nsg_ctx *ctx, const double *host);
int nsg_set_delta(nsg_ctx *ctx, const double *host);
int nsg_get_solution(nsg_ctx *ctx, double *host);
/* the ghosted vector `solution` that output() reads (cpp:697-700): owned entries then the ghost layer, n_loc doubles */
int nsg_get_solution_ghosted(nsg_ctx *ctx, double *host);
int nsg_get_delta(nsg_ctx *ctx, double *host);
int nsg_get_residual(nsg_ctx *ctx, double *host);
int nsg_get_matrix_values(nsg_ctx *ctx, double *host /* nnz(J), CSR order */);
int nsg_get_pm_values(nsg_ctx *ctx, double *host /* nnz(Mp) */);
/* The counterpart of nsg_get_solution_ghosted: writes the owned entries AND the ghost layer of `solution` as given (n_loc
 * doubles), with no exchange. Lets one GPU hold the P per-rank contexts of a partition with correct ghost values. */
int nsg_set_solution_ghosted(nsg_ctx *ctx, const double *host);

/* N3 (SURVEY 8f; the reference has no drag/lift code): force of the fluid on the body bounded by the
 * faces with `boundary_id` (13 = cylinder, cpp:368), from the current `solution`:
 * F = -oint (rho nu grad(u) n - p n) ds, n = outward normal of the fluid domain, integrated with the
 * reference's 3-point face rule (cpp:52). out2 = (drag F_x, lift F_y), global over all ranks. */
int nsg_boundary_force(nsg_ctx *ctx, int32_t boundary_id, double *out2);

/* Global cell ids (nst_part_cell_ids) and ownership flags (nst_part_cell_owned) of the n_cells local cells, for
 * nsg_eval_points. Call after nsg_set_mesh. Without it every local cell is owned and its global id is its local index,
 * which is right for P = 1. */
int nsg_set_cell_ownership(nsg_ctx *ctx, const int32_t *global_cell_id, const uint8_t *owned);

/* Point evaluation of the current `solution` (probes, the pressure difference across a body, transfer to another mesh):
 * locates the n points xy[2n] in the mesh and evaluates there u_x, u_y, p (values[3n], point-major) and, if grads is not
 * NULL, du_x/dx, du_x/dy, du_y/dx, du_y/dy, dp/dx, dp/dy (grads[6n]); cell[n] (may be NULL) gets the global id of the
 * cell used. A point lies in a cell when its three barycentric coordinates are >= -1e-12; of the owned cells containing
 * it the one with the smallest global id is used, so the result does not depend on the rank count. A point no cell
 * contains (or with a non-finite coordinate) gets cell -1 and NaN values. The spatial index (a uniform grid of bins) is
 * built on the first call. collective != 0 on a context with a communicator: every rank passes the same points and
 * receives the same results (NCCL all-reduce of the winning cell id, then of the values); otherwise each context
 * answers from its own owned cells. n = 0 does nothing; before nsg_set_mesh: NSG_ERR_STATE. */
int nsg_eval_points(nsg_ctx *ctx, int64_t n, const double *xy, int32_t collective, double *values, double *grads,
                    int64_t *cell);
/* The spatial index of nsg_eval_points (NSG_ERR_STATE before the first call): out8 = bins in x, bins in y, bin side,
 * cell entries, non-empty bins, entries of the largest bin, index bytes (8 (bins + 1) + 4 entries), build time in ms
 * (host clock, ending in a device synchronise). */
int nsg_points_index_info(nsg_ctx *ctx, double *out8);

/* Building blocks exported for parity tests and roofline measurement. x, y are host vectors of
 * owned length. nsg_spmv: y = J x (jacobian_matrix.vmult). nsg_precond_apply: y = P^-1 x for the
 * given kind with the CURRENT matrices (initialize + vmult, hpp:526-572 / 582-619).
 * nsg_ilu_apply: y = (LU)^-1 x of Ifpack ILU(0) on block which = 0 (A) or 1 (Mp). */
int nsg_spmv(nsg_ctx *ctx, const double *x, double *y);
int nsg_precond_apply(nsg_ctx *ctx, int32_t precond, const double *x, double *y);
int nsg_ilu_apply(nsg_ctx *ctx, int32_t which, const double *x, double *y);

/* Repeat a kernel `reps` times on device-resident data and return the mean time per
 * launch in milliseconds (CUDA events on the context's stream). what: 0 = assembly (cells +
 * Neumann, no Dirichlet), 1 = SpMV J*delta, 2 = add_and_dot, 3 = dot, 4 = one halo exchange, 5 = FP64 pipe
 * micro-benchmark (SM count x 16 CTAs x 256 threads x 8 chains x 2048 dependent DFMA = SMs x 67 108 864 DFMA per launch,
 * 2 flop each: the measured FP64 peak the assembly's FP64-pipe share is quoted against), 6 / 7 = one ILU(0) apply (forward +
 * backward triangular solve, tuning key 4) of the velocity / pressure-mass block, factorised before the timed region,
 * 8 = locate + evaluate the points of the last nsg_eval_points call (local mode, without the host copies). */
int nsg_time_kernel(nsg_ctx *ctx, int32_t what, int32_t reps, double *ms_per_launch);

/* Tuning knobs that do not change what is computed (only the summation order inside a row):
 * key 0 = SpMV kernel variant: 0 CSR-stream through shared memory (every row summed in CSR order, as the reference's
 * Epetra loop: the strict-parity kernel); 1 CSR-vector, 8 lanes per row; 4 = 1 with all loads of a row in flight,
 * persistent, prefetched row extents; 7 (default) = 4 serving the two rows of a velocity node together (they have the
 * same column list: one index load and one x gather feed two entries; bitwise the same result as 4). The six other
 * variants measured in round 1 (profiles/r01_summary.md) were slower and have been removed.
 * key 1 = assembly kernel variant: 0 literal 7-point quadrature loop for every term, contributions added in ascending
 * cell order as the reference's loop adds them (strict-parity kernel); 4 per-cell packets from a streaming pre-pass, one
 * (owner, cell) pair per lane, lanes sorted by commit round, first-touch stores, TMA bulk write-out (round-1 default);
 * 5 (default) the "fan" scheme, see below. Variants 1-3 of round 1 were slower and have been removed.
 * Vertex valence (cells per vertex) each one serves: 5 up to 32 on oriented manifold triangulations, 4 up to 32, 0 up to
 * 64; selecting a variant the mesh exceeds fails. A pattern built on the device (nsg_set_pattern_from_cells) holds valence
 * up to 34 inside the domain and 33 on the boundary.
 * key 3 = Gram-Schmidt variant of SolverGMRES: 0 (default) modified, the chain of add_and_dot that deal.II
 * <= 9.4 runs (SURVEY 9-8); 1 classical (h = V^T w, w -= V h: two passes and two all-reduces per step
 * instead of k+1; deal.II >= 9.5 offers it as OrthogonalizationStrategy::classical_gram_schmidt).
 * key 4 = triangular solves of the ILU(0) preconditioners: 0 one launch per dependency level; 1 one launch per
 * solve on all SMs, rows wait on the completion stamps of the rows they depend on; 2 one CTA walks the levels, rows
 * and factors stream through shared-memory rings in level order and the unknowns sit in a shared-memory window
 * (a dependency hop is a CTA barrier instead of an L2 round trip: the fast choice for the long, narrow level
 * structure of 2-D meshes); -1 (default) the library picks 1 or 2 per block from the level count and the size of
 * the factors.  All four give bitwise the same result.
 * key 5 = the whole identity-preconditioned GMRES solve as ONE cooperative kernel (vector entries in registers across
 * the Gram-Schmidt chain, one stamped-slot exchange per inner product; one rank, modified Gram-Schmidt): 0 off, 1 (default) for systems
 * of up to 65 536 unknowns (the meshes the reference ships: 2x faster there), 2 whenever the system fits (up to 148 x 256 x 8 unknowns). Same algorithm and scalars as
 * the multi-kernel path; the inner-product sums are partitioned differently (agreement to rounding, not bitwise).
 * key 2 = CUDA graphs for the launch segments of the identity-preconditioned GMRES cycle: 1 (default) on, 0 off.
 * key 1 = 5 (default since round 2): the "fan" scheme - one (owner, cell) pair per lane integrated in a rotated local
 * frame (owner = local vertex 0 / edge 0: all tables are immediates), the lanes of an owner in one warp in fan order,
 * shared-edge contributions combined by warp shuffles, every entry stored exactly once (no read-modify-write, no
 * commit rounds). Needs an oriented manifold triangulation with valence <= 32; nsg_set_mesh serves other meshes by 4
 * (valence <= 32) or else 0 (valence <= 64) automatically and fails on a vertex of more than 64 cells.
 * key 6 = L2 prefetch distances of variant 5 in chunks: records (low 16 bits, default 600), packets (high 16 bits, default 0). */
int nsg_set_tuning(nsg_ctx *ctx, int32_t key, int32_t value);

/* Counters since creation: kernel launches issued by this library, bytes it moved H2D / D2H. */
int nsg_get_counters(nsg_ctx *ctx, int64_t *launches, int64_t *h2d_bytes, int64_t *d2h_bytes);

/* Per-phase device time (ms) of the last call of each: [0] assemble, [1] dirichlet, [2] solve. */
int nsg_get_phase_ms(nsg_ctx *ctx, double *out3);

#ifdef __cplusplus
}
#endif
#endif
