// nsg_pattern.cuh — SURVEY §8f N4: the two sparsity patterns of the reference's setup() (DoFTools::make_sparsity_pattern
// with full coupling for the Jacobian, src/NavierStokesSolver.cpp:107-110, and the p-p pattern of the pressure mass
// matrix, cpp:143-158) built ON THE DEVICE from the cell -> dof table, bit-identical to the host build of libnst.so
// (nst_part_build): row r = an owned DoF, columns = the local ids of every DoF of every cell that holds r, ascending
// (= [owned u | owned p | ghost u | ghost p]).
//
// Rows come in groups: the two rows of a velocity node share one column list, a pressure vertex has one row (its
// Jacobian row and its pressure-mass row).  Pipeline: count (group, cell) incidences -> scan -> fill the group -> cells
// lists -> one thread per group merges the node keys of its cells into a sorted unique list in local memory and emits the
// row lengths -> scan -> the same merge again writes the columns.  Incidence lists are filled with atomics (their order
// is not deterministic) but every row is sorted, so the result is.  No library calls: the scans are the three small
// kernels below.
#pragma once
#include "nsg_common.cuh"

namespace nsg {

// ---- exclusive scan: out[i] = sum_{j<i} in[j], out[n] = total (int64); blocks of SCAN_B elements, recursive ----
constexpr int SCAN_B = 1024;
template <class TIn>
__global__ void __launch_bounds__(SCAN_B)
k_scan_blocks(int64_t n, const TIn *__restrict__ in, int64_t *__restrict__ out, int64_t *__restrict__ block_sums) {
  __shared__ int64_t s_w[SCAN_B / 32];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int64_t i = blockIdx.x * (int64_t)SCAN_B + t;
  const int64_t v = i < n ? (int64_t)in[i] : 0;
  int64_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_w[wid] = x;
  __syncthreads();
  if (wid == 0) {
    int64_t w = lane < SCAN_B / 32 ? s_w[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    s_w[lane] = w;  // inclusive scan of the warp totals
  }
  __syncthreads();
  const int64_t base = wid > 0 ? s_w[wid - 1] : 0;
  if (i < n) out[i] = base + x - v;  // exclusive inside the block
  if (t == SCAN_B - 1) block_sums[blockIdx.x] = base + x;
}
__global__ void k_scan_add(int64_t n, int64_t *__restrict__ out, const int64_t *__restrict__ block_off) {
  const int64_t i = blockIdx.x * (int64_t)SCAN_B + threadIdx.x;
  if (i < n) out[i] += block_off[blockIdx.x];
}
// out has n + 1 entries; tmp is scratch for the block sums of every level (>= 2 * (n / SCAN_B + 2) + 64 entries)
template <class TIn>
static int dev_exclusive_scan(nsg_ctx *c, int64_t n, const TIn *in, int64_t *out, int64_t *tmp) {
  if (n <= 0) {
    NSG_CUDA(cudaMemsetAsync(out, 0, 8, c->stream));
    return NSG_OK;
  }
  const int64_t nb = (n + SCAN_B - 1) / SCAN_B;
  int64_t *sums = tmp, *sums_scan = tmp + nb + 1;  // sums_scan gets nb + 1 entries
  k_scan_blocks<TIn><<<(unsigned)nb, SCAN_B, 0, c->stream>>>(n, in, out, sums);
  NSG_LAUNCH_CHECK(c);
  if (nb > 1) {
    NSG_TRY(dev_exclusive_scan<int64_t>(c, nb, sums, sums_scan, tmp + 2 * (nb + 1)));
    k_scan_add<<<(unsigned)nb, SCAN_B, 0, c->stream>>>(n, out, sums_scan);
    NSG_LAUNCH_CHECK(c);
    NSG_CUDA(cudaMemcpyAsync(out + n, sums_scan + nb, 8, cudaMemcpyDeviceToDevice, c->stream));
  } else {
    NSG_CUDA(cudaMemcpyAsync(out + n, sums, 8, cudaMemcpyDeviceToDevice, c->stream));
  }
  return NSG_OK;
}

// group of local slot s (0..5 velocity nodes, 6..8 pressure vertices) of a cell, or -1 if the DoF is not owned
__device__ __forceinline__ int64_t pat_group(const int32_t *__restrict__ cd, int s, int64_t n_own_u, int64_t n_own) {
  if (s < 6) {
    const int32_t d = cd[uidx(s)];
    return d < n_own_u ? d >> 1 : -1;
  }
  const int32_t d = cd[3 * (s - 6) + 2];
  return (d >= n_own_u && d < n_own) ? (n_own_u >> 1) + (d - n_own_u) : -1;
}
__global__ void k_pat_count(int64_t T, const int32_t *__restrict__ cell_dofs, int64_t n_own_u, int64_t n_own, int32_t *gcount) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= 9 * T) return;
  const int64_t cell = i / 9;
  const int64_t g = pat_group(cell_dofs + 15 * cell, (int)(i - 9 * cell), n_own_u, n_own);
  if (g >= 0) atomicAdd(gcount + g, 1);
}
__global__ void k_pat_fill(int64_t T, const int32_t *__restrict__ cell_dofs, int64_t n_own_u, int64_t n_own, const int64_t *__restrict__ gptr,
                           int32_t *cursor, int32_t *__restrict__ gcells) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= 9 * T) return;
  const int64_t cell = i / 9;
  const int64_t g = pat_group(cell_dofs + 15 * cell, (int)(i - 9 * cell), n_own_u, n_own);
  if (g >= 0) gcells[gptr[g] + atomicAdd(cursor + g, 1)] = (int32_t)cell;
}

// node keys of a patch: a vertex of valence v has 3 v + 1 velocity nodes and v + 1 vertices in its patch inside the domain,
// 3 v + 3 and v + 2 on the boundary, so the builder holds valence <= 34 inside and <= 33 on the boundary
constexpr int PAT_MAXU = 104, PAT_MAXP = 40;
// sorted unique keys of group g: velocity nodes (key = first dof id of the node) and pressure dofs of its cells
__device__ __forceinline__ bool pat_keys(int64_t g, const int64_t *__restrict__ gptr, const int32_t *__restrict__ gcells,
                                         const int32_t *__restrict__ cell_dofs, int32_t *ku, int &nu, int32_t *kp, int &np) {
  nu = np = 0;
  auto insert = [](int32_t *k, int &n, int cap, int32_t key) -> bool {
    int lo = 0, hi = n;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (k[mid] < key) lo = mid + 1;
      else hi = mid;
    }
    if (lo < n && k[lo] == key) return true;
    if (n >= cap) return false;
    for (int j = n; j > lo; --j) k[j] = k[j - 1];
    k[lo] = key;
    ++n;
    return true;
  };
  bool ok = true;
  for (int64_t p = gptr[g]; p < gptr[g + 1]; ++p) {
    const int32_t *cd = cell_dofs + 15 * (int64_t)gcells[p];
#pragma unroll
    for (int s = 0; s < 6; ++s) ok &= insert(ku, nu, PAT_MAXU, cd[uidx(s)]);
#pragma unroll
    for (int m = 0; m < 3; ++m) ok &= insert(kp, np, PAT_MAXP, cd[3 * m + 2]);
  }
  return ok;
}
// row lengths: rows 2g, 2g+1 of a velocity group and the row of a pressure group have 2 nu + np Jacobian columns; the
// pressure-mass pattern has np columns in the pressure rows and none in the velocity rows
__global__ void k_pat_rowlen(int64_t n_groups, int64_t n_ug, const int64_t *__restrict__ gptr, const int32_t *__restrict__ gcells,
                             const int32_t *__restrict__ cell_dofs, int32_t *__restrict__ rowlen, int32_t *__restrict__ pm_rowlen, int32_t *err) {
  const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  int32_t ku[PAT_MAXU], kp[PAT_MAXP];
  int nu, np;
  if (!pat_keys(g, gptr, gcells, cell_dofs, ku, nu, kp, np)) *err = 1;
  const int32_t len = 2 * nu + np;
  if (g < n_ug) {
    rowlen[2 * g] = rowlen[2 * g + 1] = len;
    pm_rowlen[2 * g] = pm_rowlen[2 * g + 1] = 0;
  } else {
    rowlen[g + n_ug] = len;
    pm_rowlen[g + n_ug] = np;
  }
}
__global__ void k_pat_cols(int64_t n_groups, int64_t n_ug, const int64_t *__restrict__ gptr, const int32_t *__restrict__ gcells,
                           const int32_t *__restrict__ cell_dofs, const int64_t *__restrict__ rowptr, int32_t *__restrict__ col,
                           const int64_t *__restrict__ pm_rowptr, int32_t *__restrict__ pm_col) {
  const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  int32_t ku[PAT_MAXU], kp[PAT_MAXP];
  int nu, np;
  pat_keys(g, gptr, gcells, cell_dofs, ku, nu, kp, np);
  const int64_t row = g < n_ug ? 2 * g : g + n_ug;
  int32_t *o0 = col + rowptr[row], *o1 = g < n_ug ? col + rowptr[row + 1] : nullptr;
  // merge by id: a velocity node's key is its first dof, it emits two columns
  int iu = 0, ip = 0, w = 0;
  while (iu < nu || ip < np) {
    if (ip >= np || (iu < nu && ku[iu] < kp[ip])) {
      o0[w] = ku[iu], o0[w + 1] = ku[iu] + 1;
      if (o1) o1[w] = ku[iu], o1[w + 1] = ku[iu] + 1;
      w += 2, ++iu;
    } else {
      o0[w] = kp[ip];
      if (o1) o1[w] = kp[ip];
      ++w, ++ip;
    }
  }
  if (g >= n_ug) {
    int32_t *m = pm_col + pm_rowptr[row];
    for (int j = 0; j < np; ++j) m[j] = kp[j];
  }
}
// groups of SpMV variant 7 that read a ghost column (columns ascend: ghosts, if any, end the row)
__global__ void k_pat_ghost_flag(int64_t n_groups, int64_t n_ug, int64_t n_own, const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                                 uint8_t *__restrict__ flag) {
  const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  const int64_t r = g < n_ug ? 2 * g : g + n_ug;
  flag[g] = (rowptr[r + 1] > rowptr[r] && col[rowptr[r + 1] - 1] >= n_own) ? 1 : 0;
}

// column offsets of the lanes of a fan list (nsg_fanlist.inl) looked up on the device: off[0..5] = position of the column
// pair of the ROTATED local node l in the owner's Jacobian row, off[6..8] = position of the three pressure columns in the
// Jacobian row (velocity owners) or in the pressure-mass row (pressure owners)
__global__ void k_fan_offsets(int kind, int64_t n_recs, int lanes_per_chunk, PairRec *__restrict__ recs, const ChunkInfo *__restrict__ chunks,
                              const int32_t *__restrict__ cell_dofs, int64_t n_own_u, const int64_t *__restrict__ rowptr,
                              const int32_t *__restrict__ col, const int64_t *__restrict__ pm_rowptr, const int32_t *__restrict__ pm_col, int32_t *err) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_recs) return;
  PairRec rc = recs[i];
  if (rc.cell < 0) return;
  const ChunkInfo &ci = chunks[i / lanes_per_chunk];
  const uint32_t kw = (uint32_t)rc.k;
  const int kc = (int)(kw & 7u), gl = (int)((kw >> 16) & 255u);
  const int r = kc >= 3 ? kc - 3 : kc;
  const int64_t g = ci.g0 + gl;
  const int64_t row = kind == 0 ? 2 * g : n_own_u + g;
  const int32_t *cd = cell_dofs + 15 * (int64_t)rc.cell;
  auto find = [&](const int32_t *base, int64_t s, int64_t e, int32_t key) -> int {
    int64_t lo = s, hi = e;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (base[mid] < key) lo = mid + 1;
      else hi = mid;
    }
    if (lo >= e || base[lo] != key) {
      *err = 1;
      return 0;
    }
    return (int)(lo - s);
  };
  const int64_t rs = rowptr[row], re = rowptr[row + 1];
#pragma unroll
  for (int l = 0; l < 6; ++l) {
    const int lc = l < 3 ? (l + r) % 3 : 3 + (l - 3 + r) % 3;
    rc.off[l] = (uint16_t)find(col, rs, re, cd[uidx(lc)]);
  }
#pragma unroll
  for (int m = 0; m < 3; ++m) {
    const int32_t key = cd[3 * ((m + r) % 3) + 2];
    rc.off[6 + m] = kind == 0 ? (uint16_t)find(col, rs, re, key) : (uint16_t)find(pm_col, pm_rowptr[row], pm_rowptr[row + 1], key);
  }
  recs[i] = rc;
}

}  // namespace nsg
