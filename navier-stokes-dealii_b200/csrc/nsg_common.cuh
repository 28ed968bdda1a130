// nsg_common.cuh — context, error handling and small helpers shared by the libnsg.so sources.
#pragma once
#include <cuda_runtime.h>
#include "nsg_nccl.cuh"
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/nsg.h"

namespace nsg {

extern thread_local std::string g_err;
int fail(int code, const std::string &msg);

#define NSG_CUDA(expr)                                                                          \
  do {                                                                                          \
    cudaError_t e__ = (expr);                                                                   \
    if (e__ != cudaSuccess)                                                                     \
      return ::nsg::fail(NSG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));    \
  } while (0)
#define NSG_NCCL(expr)                                                                          \
  do {                                                                                          \
    ncclResult_t r__ = (expr);                                                                  \
    if (r__ != ncclSuccess)                                                                     \
      return ::nsg::fail(NSG_ERR_NCCL, std::string(#expr) + ": " + ::nsg::nccl_api().GetErrorString(r__)); \
  } while (0)
#define NSG_TRY(expr)          \
  do {                         \
    int rc__ = (expr);         \
    if (rc__ != NSG_OK) return rc__; \
  } while (0)
#define NSG_LAUNCH_CHECK(ctx)  \
  do {                         \
    (ctx)->launches++;         \
    NSG_CUDA(cudaGetLastError()); \
  } while (0)

// One (row-owner, cell) work item of the assembly: `k` is the local scalar index of the owner's
// node in the cell (P2 index 0..5 for a velocity node, P1 index 0..2 for a pressure row);
// off[0..5] = offset inside the owner's Jacobian row of the column pair (2m,2m+1) of the cell's
// six P2 nodes; off[6..8] = offset of the cell's three pressure columns (in the Jacobian row for a
// velocity owner, in the pressure-mass row for a pressure owner).
struct __align__(16) PairRec {
  int32_t cell;
  int32_t k;
  uint16_t off[12];
};
static_assert(sizeof(PairRec) == 32, "PairRec must be 32 bytes");

// Row-owner work lists.  An owner (velocity node = 2 rows, or pressure row) with a patch of s cells
// is served by ceil(s/PPT) thread "slots"; slot r integrates pairs r, r+nslots, ... so every thread
// does at most PPT (owner, cell) pairs and the CTA is balanced.  Slots of one owner commit their
// local rows to the shared chunk image in rounds (slot 0, barrier, slot 1, ...), i.e. in ascending
// cell order: no atomics, fixed summation order.
constexpr int ASM_PPT = 2;
constexpr int64_t ASM_STAGE_CAP = int64_t(1) << 30;  // max staged entries per chunk (env NSG_ASM_STAGE_CAP overrides)
struct __align__(16) ChunkInfo {
  int32_t g0, g1;        // owners [g0,g1) of this chunk (consecutive rows)
  int32_t n_threads;     // sum of slots (<= NPC)
  int32_t max_slots;     // commit rounds
  int64_t rec_base;      // records of iteration j, thread t at rec_base + j*n_threads + t
  // everything the packet-based kernels (variant 2) need without a dependent row-pointer load:
  int64_t rs;            // first Jacobian entry of the chunk's rows
  int64_t ms;            // first pressure-mass entry (pressure chunks)
  int32_t cnt, mcnt;     // number of Jacobian / pressure-mass entries of the chunk
  int64_t pad;
};
static_assert(sizeof(ChunkInfo) == 64, "ChunkInfo layout");
struct WorkList {
  int64_t n_groups = 0, n_chunks = 0, n_pairs = 0, n_recs = 0;
  ChunkInfo *chunks = nullptr;   // [n_chunks]
  uint16_t *tdesc = nullptr;     // [n_chunks*NPC] owner index inside the chunk | slot << 8
  uint2 *tdesc3 = nullptr;       // [n_chunks*NPC] x = offset of the owner's first row in the chunk image (pressure: x =
                                 // J-row offset | mass-row offset << 16); y = row length | slot << 16 | owner << 24;
                                 // y = 0xffffffff marks a padding lane
  PairRec *recs = nullptr;       // [n_recs]; cell = -1 marks "no work"
  int64_t max_stage = 0;         // max number of staged matrix entries of a chunk
};

// Peer memory over NVLink (CUDA IPC): every rank owns ONE mailbox allocation that all peers map:
//   [ all-reduce words | halo table | halo inbox ]
// Every datum travels as a 16-byte {value, sequence stamp} word written by one 128-bit store and read by one 128-bit
// load: the stamp arrives with the value, so neither side needs a fence, a separate flag or a second round trip.
//
// One-shot all-reduce, fused into the tail of the reduction kernels: reduction number s writes my partial value(s) into
// slot [s&1][my rank] of EVERY rank's mailbox, then polls the P slots of my own mailbox until they carry stamp s and
// adds the P values in rank order - every rank gets the bit-identical sum, with no host or NCCL call on the critical
// path of the k+1 dependent reductions of a GMRES step.  (Parity double-buffering is safe: nobody can start s+2
// before everybody has finished reading s.)
//
// Halo exchange (the Epetra Import behind every vmult, cpp:583,587,618): the owner of a DoF stores {value, stamp} straight
// into the inbox of each neighbour that holds it as a ghost (k_halo_push); the neighbour polls its own inbox and scatters
// into the ghost range (k_halo_wait_scatter).  The inbox interleaves the two parities ([slot][parity]).
constexpr int PEER_MAX_RANKS = 16;
constexpr int PEER_MAX_VALS = 32;
struct __align__(16) PeerWord {
  double v;
  unsigned long long seq;
};
static_assert(sizeof(PeerWord) == 16, "PeerWord layout");
constexpr int64_t PEER_AR_WORDS = 2ll * PEER_MAX_RANKS * PEER_MAX_VALS;  // [parity][source rank][value]
struct PeerHaloTable {                                                   // what a sender needs to know about my inbox
  int64_t recv_off[PEER_MAX_RANKS];  // first inbox slot of source rank q (-1: not a neighbour)
  int64_t recv_cnt[PEER_MAX_RANKS];
};
constexpr int64_t PEER_TABLE_BYTES = 256;
static_assert(sizeof(PeerHaloTable) <= PEER_TABLE_BYTES, "halo table");
constexpr int64_t PEER_INBOX_OFFSET = PEER_AR_WORDS * 16 + PEER_TABLE_BYTES;  // bytes
constexpr long long PEER_TIMEOUT_CYCLES = 60000000000ll;  // ~30 s at 1.9 GHz: bounded, so a lost peer cannot hang the GPU
struct PeerComm {
  PeerWord *ar[PEER_MAX_RANKS];   // ar[p] = all-reduce words of rank p's mailbox
  unsigned long long *seq_ctr;    // this rank's count of completed fused reductions (device memory)
  int rank, n_ranks;
};

// deal.II SolverGMRES bookkeeping kept on the device (SURVEY §9-8)
constexpr int GM_MAX_TMP = 64;
struct GmresCtl {
  // header (first 64 bytes are mirrored to the host at the synchronisation points)
  double tol, rho, nrm2, norm_start2, inv_s;
  int32_t state;  // 0 iterate, 1 success, 2 failure; | 0x100 when decided inside a cycle
  int32_t accumulated, dim, max_steps, n_tmp, hist_cap;
  double gamma[GM_MAX_TMP], ci[GM_MAX_TMP], si[GM_MAX_TMP], h[GM_MAX_TMP], h2[GM_MAX_TMP], y[GM_MAX_TMP];
  double H[GM_MAX_TMP * GM_MAX_TMP];
};
constexpr size_t GM_HEADER_BYTES = 64;

// One cached CUDA graph per launch segment of the identity-preconditioned restart cycle (the stretches
// between two host synchronisation points).  Small meshes are launch-bound (~19 kernels per GMRES step);
// replaying a captured segment costs a fraction of issuing its kernels one by one.
struct GraphKey {
  int seg, n_tmp;
  int64_t n, off;
  const void *x, *b, *basis, *hist;
  bool operator==(const GraphKey &o) const {
    return seg == o.seg && n_tmp == o.n_tmp && n == o.n && off == o.off && x == o.x && b == o.b && basis == o.basis && hist == o.hist;
  }
};
struct GraphEntry {
  GraphKey key;
  cudaGraphExec_t exec;
  int64_t launches;
};

struct CsrBlock {  // a sub-matrix held separately (A, Mp, B of the block preconditioners)
  int64_t n = 0, nnz = 0;
  int64_t *rowptr = nullptr;
  int32_t *col = nullptr;
  double *val = nullptr;
  int64_t *src = nullptr;   // position of each entry in the parent CSR (for the value refresh)
  int64_t *diag = nullptr;  // position of the diagonal in each row
  // level schedule of the lower / upper triangular solves and of the ILU(0) elimination
  int32_t n_levels = 0, n_ulevels = 0;
  int32_t *level_rows = nullptr, *ulevel_rows = nullptr;  // [n] rows sorted by forward / backward level
  std::vector<int32_t> h_level_ptr, h_ulevel_ptr;         // [n_levels+1] on the host (launch bounds)
  double *fval = nullptr;  // ILU(0) factors on the same pattern
  double *dinv = nullptr;
  int32_t *chunk_rows = nullptr;
  int64_t n_chunks = 0;
  // single-launch ("sync-free") triangular solves: per-row completion stamps + ticket counter for the CTA order
  ulonglong2 *done_l = nullptr, *done_u = nullptr;    // [n] {value, epoch stamp} of the forward / backward unknowns
  unsigned long long *ticket = nullptr;               // [2] monotone counters (forward, backward)
  unsigned long long epoch = 0;
  unsigned long long tickets_l = 0, tickets_u = 0;    // host mirror: tickets handed out so far
  int32_t *sf_error = nullptr;                        // set if a wait ran into its time limit
  // one-CTA triangular solves (tuning key 4 = 2): rows, entries and unknowns stored in level order ("positions"), so the
  // kernel streams them through shared-memory rings and a dependency hop is a CTA barrier, not an L2 round trip
  struct Tri {
    int32_t n_levels = 0;
    int64_t nq = 0;             // slots (entries incl. padding)
    int4 *info = nullptr;       // [n_levels+1] {first slot, slabs per group, 1 = staged through the rings / 0 = read in place, first position}
    int4 *slots = nullptr;      // [nq] {factor (refreshed after every factorisation), position of the entry's unknown or ~position
                                //       once it has left the shared-memory window, 0}
    int64_t *fsrc = nullptr;    // [nq] where the entry sits in fval; -1 = padding
    int32_t *rowid = nullptr;   // [n] row index of each position
    int32_t *ra_src = nullptr;  // [n] forward: row index (gathers the right-hand side); backward: position in the forward layout
    double2 *rows = nullptr;    // [n] by position: {gathered right-hand side, inverse pivot}
    double *yg = nullptr;       // [n] unknowns by position
  } triL, triU;
  bool tri_ok = false;          // the layouts exist (block small enough for 32-bit entry indices)
  bool tri_pick = false;        // ... and the one-CTA solve is estimated faster than the stamped single launch
};

}  // namespace nsg

struct nsg_ctx {
  int device = 0;
  cudaStream_t stream = nullptr, own_stream = nullptr;
  // sizes
  int64_t n_own_u = 0, n_own_p = 0, n_own = 0, n_ghost_u = 0, n_ghost_p = 0, n_loc = 0, stride = 0;
  int64_t nnz = 0, pm_nnz = 0;
  int64_t n_cells = 0, n_vertices = 0, n_bfaces = 0;
  bool have_pattern = false, have_mesh = false;
  bool pattern_on_device = false;  // built by nsg_set_pattern_from_cells: no host copy of the column indices exists
  nsg_params prm{};
  // host copies of the patterns kept until nsg_set_mesh has built the work lists
  std::vector<int64_t> h_rowptr, h_pm_rowptr;
  std::vector<int32_t> h_col, h_pm_col;
  // device CSR
  int64_t *rowptr = nullptr, *pm_rowptr = nullptr;
  int32_t *col = nullptr, *pm_col = nullptr;
  double *vals = nullptr, *pm_vals = nullptr;
  int32_t *spmv_chunk_rows = nullptr;
  int64_t *diag_pos = nullptr;
  unsigned long long *first_idx = nullptr;
  int spmv_variant = 0, asm_variant = 5;
  int gmres_fused = 1;  // tuning key 5: 0 off, 1 systems up to gmres_fused_max_n unknowns, 2 whenever the vectors fit the grid's registers
  int64_t gmres_fused_max_n = 65536;  // measured: 2.0x faster at 29 646 unknowns, 1.08x at 117 324, 0.86x at 232 003
  double *gf_partials = nullptr;
  int ilu_variant = -1;  // -1: choose per block (1 or 2); 0: one launch per dependency level; 1: single launch, rows wait on
                         // completion stamps; 2: one CTA, level order, unknowns in a shared-memory window
  bool use_graphs = true;
  int orthogonalization = 0;  // 0 modified Gram-Schmidt (deal.II <= 9.4 default), 1 classical
  std::vector<nsg::GraphEntry> graphs;
  int32_t last_solve[4] = {0, 0, 0, 0};  // nsg_last_solve_info
  bool have_paired = false;  // rows 2g, 2g+1 of every velocity node have the same column list (SpMV variant 7)
  int64_t spmv_n_chunks = 0;
  // mesh
  double *geom = nullptr;  // [5T] J^-T (a00,a01,a10,a11), |det J|
  double *geom8 = nullptr;  // [8T] grad lambda_0..2, |det J|, 0 (assembly variant 5)
  double *cellpk = nullptr;  // [44T] per-cell packets of assembly variant 2 (rewritten by every nsg_assemble)
  double *xy = nullptr;
  int32_t *cell_vertices = nullptr, *cell_dofs = nullptr;
  nsg::WorkList wl_u, wl_p;
  nsg::WorkList wl_u5, wl_p5;  // assembly variant 4: one pair per lane, lanes sorted by (round, cell)
  nsg::WorkList wl_u6, wl_p6;  // assembly variant 5 ("fan"): the lanes of an owner in one warp, every entry stored once
  int asm_pf_rec = 600, asm_pf_pk = 0;  // variant 5: L2 prefetch distances in chunks (tuning key 6; measured: records 600 ahead -3 %)
  bool fan_ok = false;         // the mesh is an oriented manifold triangulation the fan scheme can serve
  // The pressure rows of J (B and the zero p-p block) and all of Mp hold what the pressure-row kernel of asm_variant
  // computes from the geometry and nu: launch_assembly skips that kernel while this is set.  Cleared by nsg_set_params
  // when nu changes, by nsg_apply_dirichlet when it constrains a pressure row and by nsg_set_tuning when the assembly
  // variant changes (the variants sum in different orders).  Pattern and mesh are set once, before the first assembly.
  // Per context: with several ranks each context holds only its owned pressure rows.
  bool p_rows_valid = false;
  // Neumann: boundary nodes -> faces
  int64_t n_bnodes = 0;
  int32_t *bnode_dof = nullptr, *bnode_ptr = nullptr, *bnode_face = nullptr, *bnode_pos = nullptr;
  int32_t *bface_cell = nullptr, *bface_face = nullptr, *bface_tag = nullptr;
  // vectors (stride doubles each; ghosts at [n_own, n_loc))
  double *sol = nullptr, *sol_old = nullptr, *delta = nullptr, *R = nullptr;
  double *basis = nullptr;  // n_tmp * stride
  int32_t basis_n_tmp = 0;
  double *work = nullptr;   // scratch vectors for the preconditioners (8 * stride)
  // reductions / control
  double *partials = nullptr, *partials_k = nullptr;
  unsigned int *ticket = nullptr;
  double *scal = nullptr;  // misc device scalars
  nsg::GmresCtl *ctl = nullptr, *h_ctl = nullptr;  // device / pinned host mirror
  double *hist = nullptr;
  int64_t hist_cap = 0;
  std::vector<double> h_hist;
  // Dirichlet scratch
  int32_t *dir_dofs = nullptr;
  double *dir_vals = nullptr;
  int64_t dir_cap = 0;
  std::vector<int32_t> h_dir_dofs;  // what dir_dofs / dir_vals hold (host copies: an unchanged list is not uploaded again)
  std::vector<double> h_dir_vals;
  // halo
  int32_t n_neighbors = 0;
  std::vector<int32_t> neighbors;
  std::vector<int64_t> send_ptr, recv_ptr;
  int32_t *send_idx = nullptr, *recv_idx = nullptr;
  double *send_buf = nullptr, *recv_buf = nullptr;
  int64_t n_send = 0, n_recv = 0;
  ncclComm_t comm = nullptr;
  int rank = 0, n_ranks = 1;
  char *mailbox = nullptr;               // this rank's mailbox (peer-writable): all-reduce words, halo table, halo inbox
  int64_t mailbox_bytes = 0;
  // peer-store halo exchange (after nsg_comm_set_peers): per send entry the destination word in the neighbour's inbox
  bool halo_peer = false;
  nsg::PeerWord **send_dst = nullptr;    // [n_send] parity-0 word; parity 1 is the next word
  unsigned long long *halo_ctr = nullptr;  // [0] pushes completed, [1] receives completed (device)
  unsigned int *halo_ticket = nullptr;     // [2]
  int32_t *halo_err = nullptr;
  int32_t *bgroups = nullptr;            // SpMV variant 7: row groups with a ghost column (recomputed after the exchange)
  int64_t n_bgroups = 0;
  nsg::PeerComm peer{};                  // n_ranks <= 1 until nsg_comm_set_peers
  unsigned long long *ar_seq = nullptr;  // device counter behind peer.seq_ctr
  void *peer_mapped[nsg::PEER_MAX_RANKS] = {};
  // block preconditioner state
  nsg::CsrBlock blkA, blkM;
  bool have_blocks = false, blocks_stale = true;
  double *inner_basis = nullptr;
  nsg::GmresCtl *inner_ctl = nullptr, *h_inner_ctl = nullptr;
  int64_t inner_its = 0;
  // staging + counters
  double *h_pinned = nullptr;
  int64_t h_pinned_cap = 0;
  int64_t launches = 0, h2d = 0, d2h = 0;
  double phase_ms[3] = {0, 0, 0};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaStream_t aux_stream = nullptr;  // pressure-row assembly runs beside the velocity rows
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};
