// nsg_points.cuh — point location and evaluation of the P2-P1 solution at arbitrary points (nsg_eval_points).
//
// Spatial index: a uniform grid of square bins over the bounding box of the context's cells, bin side
// h = sqrt(2 * mean cell area), so that a bin covers about two cells.  Every cell is listed in each bin its bounding box
// (padded by PT_PAD of its size) overlaps: count, exclusive scan, fill.  The order inside a bin follows the atomic cursor
// and is not fixed, which is harmless: the located cell does not depend on it (tie rule below).  Built on the first
// evaluation and never again (pattern and mesh are fixed for the life of a context).
//
// Locate: a point lies in a cell when its three barycentric coordinates are >= -PT_TOL.  Of all owned cells that contain
// it, the one with the smallest GLOBAL cell id wins, so the result is the same for any bin order, thread schedule and
// rank count.  Evaluate: u_x, u_y, p (and optionally their gradients) of the chosen cell, in a fixed operation order.
#pragma once
#include "nsg_common.cuh"

namespace nsg {

constexpr double PT_TOL = 1e-12;      // barycentric tolerance of the containment test
constexpr double PT_PAD = 1e-9;       // relative padding of the cell boxes: covers every point the tolerance accepts
constexpr int32_t PT_NONE = 0x7fffffff;  // "no cell" in the global-id min-reduction
constexpr int PT_RED_BLOCKS = 512;

// partials[5*b + ...] = min x, min y, -max x, -max y, sum |det J|/2 of the cells of block b
__global__ void k_pt_bbox(int64_t T, const double *__restrict__ xy, const int32_t *__restrict__ cv, const double *__restrict__ geom8,
                          double *__restrict__ partials) {
  __shared__ double s[5][256];
  double v[5] = {INFINITY, INFINITY, INFINITY, INFINITY, 0.0};
  for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < T; c += (int64_t)gridDim.x * blockDim.x) {
    for (int k = 0; k < 3; ++k) {
      const int32_t q = cv[3 * c + k];
      v[0] = fmin(v[0], xy[2 * q]), v[1] = fmin(v[1], xy[2 * q + 1]);
      v[2] = fmin(v[2], -xy[2 * q]), v[3] = fmin(v[3], -xy[2 * q + 1]);
    }
    v[4] += 0.5 * geom8[8 * c + 6];
  }
  for (int k = 0; k < 5; ++k) s[k][threadIdx.x] = v[k];
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) {
      for (int k = 0; k < 4; ++k) s[k][threadIdx.x] = fmin(s[k][threadIdx.x], s[k][threadIdx.x + w]);
      s[4][threadIdx.x] += s[4][threadIdx.x + w];
    }
    __syncthreads();
  }
  if (threadIdx.x < 5) partials[5 * blockIdx.x + threadIdx.x] = s[threadIdx.x][0];
}

__device__ inline int32_t pt_bin_coord(double v, double v0, double inv_h, int32_t n) {
  const double f = floor((v - v0) * inv_h);
  return (int32_t)fmin(fmax(f, 0.0), (double)(n - 1));
}

// mode 0: count the entries of every bin; mode 1: write them (start[] = exclusive scan of the counts, cursor[] zeroed)
template <int MODE>
__global__ void k_pt_bin_cells(int64_t T, const double *__restrict__ xy, const int32_t *__restrict__ cv, const PtGrid g,
                               int32_t *__restrict__ cnt_or_cursor, const int64_t *__restrict__ start, int32_t *__restrict__ entries) {
  for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < T; c += (int64_t)gridDim.x * blockDim.x) {
    double lo_x = INFINITY, lo_y = INFINITY, hi_x = -INFINITY, hi_y = -INFINITY;
    for (int k = 0; k < 3; ++k) {
      const int32_t q = cv[3 * c + k];
      lo_x = fmin(lo_x, xy[2 * q]), hi_x = fmax(hi_x, xy[2 * q]);
      lo_y = fmin(lo_y, xy[2 * q + 1]), hi_y = fmax(hi_y, xy[2 * q + 1]);
    }
    const double pad = PT_PAD * ((hi_x - lo_x) + (hi_y - lo_y));
    const int32_t ix0 = pt_bin_coord(lo_x - pad, g.x0, g.inv_h, g.nx), ix1 = pt_bin_coord(hi_x + pad, g.x0, g.inv_h, g.nx);
    const int32_t iy0 = pt_bin_coord(lo_y - pad, g.y0, g.inv_h, g.ny), iy1 = pt_bin_coord(hi_y + pad, g.y0, g.inv_h, g.ny);
    for (int32_t iy = iy0; iy <= iy1; ++iy)
      for (int32_t ix = ix0; ix <= ix1; ++ix) {
        const int64_t b = (int64_t)iy * g.nx + ix;
        const int32_t pos = atomicAdd(cnt_or_cursor + b, 1);
        if (MODE == 1) entries[start[b] + pos] = (int32_t)c;
      }
  }
}

// Exclusive scan of int32 counts into int64 starts (n + 1 entries), in three passes over segments of PT_SCAN_SEG counts.
constexpr int PT_SCAN_THREADS = 256, PT_SCAN_PER = 8, PT_SCAN_SEG = PT_SCAN_THREADS * PT_SCAN_PER;
__device__ inline int64_t pt_block_exclusive(int64_t v, int64_t *s_tmp, int64_t *total) {
  // Hillis-Steele over the block: v -> sum of the values of the threads before this one
  s_tmp[threadIdx.x] = v;
  __syncthreads();
  for (int w = 1; w < PT_SCAN_THREADS; w <<= 1) {
    const int64_t add = threadIdx.x >= (unsigned)w ? s_tmp[threadIdx.x - w] : 0;
    __syncthreads();
    s_tmp[threadIdx.x] += add;
    __syncthreads();
  }
  const int64_t incl = s_tmp[threadIdx.x];
  *total = s_tmp[PT_SCAN_THREADS - 1];
  __syncthreads();
  return incl - v;
}
__global__ void __launch_bounds__(PT_SCAN_THREADS) k_pt_scan_sums(int64_t n, const int32_t *__restrict__ cnt, int64_t *__restrict__ seg_sum) {
  __shared__ int64_t s[PT_SCAN_THREADS];
  const int64_t base = (int64_t)blockIdx.x * PT_SCAN_SEG + threadIdx.x * PT_SCAN_PER;
  int64_t v = 0;
  for (int k = 0; k < PT_SCAN_PER; ++k)
    if (base + k < n) v += cnt[base + k];
  int64_t total;
  pt_block_exclusive(v, s, &total);
  if (threadIdx.x == 0) seg_sum[blockIdx.x] = total;
}
__global__ void __launch_bounds__(PT_SCAN_THREADS) k_pt_scan_top(int64_t n_seg, int64_t *__restrict__ seg_sum) {
  __shared__ int64_t s[PT_SCAN_THREADS];
  int64_t carry = 0;
  for (int64_t b0 = 0; b0 < n_seg; b0 += PT_SCAN_THREADS) {
    const int64_t i = b0 + threadIdx.x;
    const int64_t v = i < n_seg ? seg_sum[i] : 0;
    int64_t total;
    const int64_t ex = pt_block_exclusive(v, s, &total);
    if (i < n_seg) seg_sum[i] = carry + ex;
    carry += total;
  }
}
__global__ void __launch_bounds__(PT_SCAN_THREADS) k_pt_scan_apply(int64_t n, const int32_t *__restrict__ cnt, const int64_t *__restrict__ seg_off,
                                                                   int64_t *__restrict__ start) {
  __shared__ int64_t s[PT_SCAN_THREADS];
  const int64_t base = (int64_t)blockIdx.x * PT_SCAN_SEG + threadIdx.x * PT_SCAN_PER;
  int64_t v = 0;
  for (int k = 0; k < PT_SCAN_PER; ++k)
    if (base + k < n) v += cnt[base + k];
  int64_t total;
  int64_t run = seg_off[blockIdx.x] + pt_block_exclusive(v, s, &total);
  for (int k = 0; k < PT_SCAN_PER; ++k)
    if (base + k < n) start[base + k] = run, run += cnt[base + k];
  if (base < n && base + PT_SCAN_PER >= n) start[n] = run;  // the thread holding the last count writes the total
}

// occupancy of the bins: stats[0] = non-empty bins, stats[1] = entries of the largest bin (both zeroed by the caller)
__global__ void k_pt_bin_stats(int64_t nb, const int32_t *__restrict__ cnt, unsigned long long *__restrict__ stats) {
  unsigned long long nonempty = 0;
  int32_t mx = 0;
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < nb; b += (int64_t)gridDim.x * blockDim.x) {
    const int32_t v = cnt[b];
    nonempty += v > 0;
    mx = max(mx, v);
  }
  for (int o = 16; o > 0; o >>= 1) {
    nonempty += __shfl_down_sync(0xffffffffu, nonempty, o);
    mx = max(mx, __shfl_down_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) {
    if (nonempty) atomicAdd(stats, nonempty);
    if (mx) atomicMax(stats + 1, (unsigned long long)mx);
  }
}

// barycentric coordinates of (px, py) in cell c: lambda_1, lambda_2 from grad lambda (geom8) and vertex 0, lambda_0 = 1 - both
__device__ inline void pt_bary(int64_t c, double px, double py, const double *__restrict__ xy, const int32_t *__restrict__ cv,
                               const double *__restrict__ geom8, double l[3]) {
  const double *g = geom8 + 8 * c;
  const int32_t v0 = cv[3 * c];
  const double dx = px - xy[2 * v0], dy = py - xy[2 * v0 + 1];
  l[1] = g[2] * dx + g[3] * dy;
  l[2] = g[4] * dx + g[5] * dy;
  l[0] = 1.0 - l[1] - l[2];
}

// One thread per point: the owned cell of smallest global id that contains it (PT_NONE: none), and its local index.
__global__ void k_pt_locate(int64_t n, const double *__restrict__ pxy, const PtGrid g, const int64_t *__restrict__ start,
                            const int32_t *__restrict__ entries, const double *__restrict__ xy, const int32_t *__restrict__ cv,
                            const double *__restrict__ geom8, const int32_t *__restrict__ gid, const uint8_t *__restrict__ owned,
                            int32_t *__restrict__ best_gid, int32_t *__restrict__ best_loc) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double px = pxy[2 * i], py = pxy[2 * i + 1];
    int32_t bg = PT_NONE, bl = -1;
    if (isfinite(px) && isfinite(py)) {
      const double fx = floor((px - g.x0) * g.inv_h), fy = floor((py - g.y0) * g.inv_h);
      if (fx >= 0.0 && fy >= 0.0 && fx < (double)g.nx && fy < (double)g.ny) {
        const int64_t b = (int64_t)fy * g.nx + (int64_t)fx;
        for (int64_t e = start[b], e1 = start[b + 1]; e < e1; ++e) {
          const int32_t c = entries[e];
          if (owned && !owned[c]) continue;
          const int32_t cg = gid ? gid[c] : c;
          if (cg >= bg) continue;
          double l[3];
          pt_bary(c, px, py, xy, cv, geom8, l);
          if (l[0] >= -PT_TOL && l[1] >= -PT_TOL && l[2] >= -PT_TOL) bg = cg, bl = c;
        }
      }
    }
    best_gid[i] = bg;
    best_loc[i] = bl;
  }
}

// One thread per point: values (and gradients) from the cell this rank located, if its global id is the winner `win_gid`
// (in local mode win_gid == best_gid).  Points no rank found get NaN; points another rank won get -0.0, the identity of the
// sum that combines the ranks (x + -0.0 == x for every x, -0.0 included), so the combined result is bitwise the winner's.
__global__ void k_pt_eval(int64_t n, const double *__restrict__ pxy, const int32_t *__restrict__ best_gid, const int32_t *__restrict__ best_loc,
                          const int32_t *__restrict__ win_gid, const double *__restrict__ xy, const int32_t *__restrict__ cv,
                          const double *__restrict__ geom8, const int32_t *__restrict__ cell_dofs, const double *__restrict__ sol,
                          double *__restrict__ vals, double *__restrict__ grads, int64_t *__restrict__ cell_out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t w = win_gid[i];
    if (cell_out) cell_out[i] = w == PT_NONE ? -1 : (int64_t)w;
    if (w == PT_NONE || best_gid[i] != w) {
      const double f = w == PT_NONE ? __longlong_as_double(0x7ff8000000000000ll) : -0.0;
      for (int k = 0; k < 3; ++k) vals[3 * i + k] = f;
      if (grads)
        for (int k = 0; k < 6; ++k) grads[6 * i + k] = f;
      continue;
    }
    const int64_t c = best_loc[i];
    double l[3];
    pt_bary(c, pxy[2 * i], pxy[2 * i + 1], xy, cv, geom8, l);
    const int32_t *cd = cell_dofs + 15 * c;
    // FE_SimplexP(2) in the order of k_face_force: vertices 0..2, then the edges (0 1), (1 2), (2 0)
    const double psi[6] = {l[0] * (2 * l[0] - 1), l[1] * (2 * l[1] - 1), l[2] * (2 * l[2] - 1),
                           4 * l[0] * l[1],       4 * l[1] * l[2],       4 * l[2] * l[0]};
    double ux = 0.0, uy = 0.0;
    for (int k = 0; k < 6; ++k) {
      const int32_t d = cd[uidx(k)];
      ux += psi[k] * sol[d];
      uy += psi[k] * sol[d + 1];
    }
    const double p0 = sol[cd[2]], p1 = sol[cd[5]], p2 = sol[cd[8]];
    vals[3 * i] = ux;
    vals[3 * i + 1] = uy;
    vals[3 * i + 2] = p0 * l[0] + p1 * l[1] + p2 * l[2];
    if (grads) {
      const double *gl = geom8 + 8 * c;  // grad lambda_0, lambda_1, lambda_2
      const double dl[3][2] = {{gl[0], gl[1]}, {gl[2], gl[3]}, {gl[4], gl[5]}};
      double out[6] = {0, 0, 0, 0, 0, 0};
      for (int j = 0; j < 2; ++j) {
        const double dpsi[6] = {(4 * l[0] - 1) * dl[0][j], (4 * l[1] - 1) * dl[1][j], (4 * l[2] - 1) * dl[2][j],
                                4 * (l[0] * dl[1][j] + l[1] * dl[0][j]), 4 * (l[1] * dl[2][j] + l[2] * dl[1][j]),
                                4 * (l[2] * dl[0][j] + l[0] * dl[2][j])};
        for (int k = 0; k < 6; ++k) {
          const int32_t d = cd[uidx(k)];
          out[j] += dpsi[k] * sol[d];
          out[2 + j] += dpsi[k] * sol[d + 1];
        }
        out[4 + j] = p0 * dl[0][j] + p1 * dl[1][j] + p2 * dl[2][j];
      }
      for (int k = 0; k < 6; ++k) grads[6 * i + k] = out[k];
    }
  }
}

// ---- host side --------------------------------------------------------------------------------------------------------
static int pt_build_index(nsg_ctx *c) {
  PointIndex &P = c->pidx;
  const double t0 = omp_get_wtime();
  const int64_t T = c->n_cells;
  double lo_x = 0, lo_y = 0, hi_x = 0, hi_y = 0, area = 0;
  if (T > 0) {
    double *part = nullptr;
    NSG_TRY(dev_alloc(&part, 5 * PT_RED_BLOCKS));
    k_pt_bbox<<<PT_RED_BLOCKS, 256, 0, c->stream>>>(T, c->xy, c->cell_vertices, c->geom8, part);
    NSG_LAUNCH_CHECK(c);
    std::vector<double> h(5 * PT_RED_BLOCKS);
    NSG_CUDA(cudaMemcpyAsync(h.data(), part, h.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    NSG_CUDA(cudaStreamSynchronize(c->stream));
    dev_free(part);
    lo_x = lo_y = hi_x = hi_y = INFINITY;
    for (int b = 0; b < PT_RED_BLOCKS; ++b) {
      lo_x = std::min(lo_x, h[5 * b]), lo_y = std::min(lo_y, h[5 * b + 1]);
      hi_x = std::min(hi_x, h[5 * b + 2]), hi_y = std::min(hi_y, h[5 * b + 3]);
      area += h[5 * b + 4];
    }
    hi_x = -hi_x, hi_y = -hi_y;
  }
  const double pad = PT_PAD * ((hi_x - lo_x) + (hi_y - lo_y)) + 1e-300;
  const double wx = hi_x - lo_x + 2 * pad, wy = hi_y - lo_y + 2 * pad;
  double h = T > 0 ? std::sqrt(2.0 * area / (double)T) : 1.0;
  if (!(h > 0)) h = std::max(wx, wy);
  // keep the grid within 2^30 bins (a degenerate mesh of slivers could ask for more)
  while ((std::floor(wx / h) + 1) * (std::floor(wy / h) + 1) > double(1 << 30)) h *= 2;
  P.grid.x0 = lo_x - pad, P.grid.y0 = lo_y - pad, P.grid.inv_h = 1.0 / h;
  P.grid.nx = (int32_t)std::floor(wx / h) + 1, P.grid.ny = (int32_t)std::floor(wy / h) + 1;
  P.h = h;
  const int64_t nb = (int64_t)P.grid.nx * P.grid.ny;
  int32_t *cnt = nullptr;
  NSG_TRY(dev_alloc(&cnt, nb));
  NSG_CUDA(cudaMemsetAsync(cnt, 0, 4 * (size_t)nb, c->stream));
  const int grid = grid_for(T, 256);
  if (T > 0) {
    k_pt_bin_cells<0><<<grid, 256, 0, c->stream>>>(T, c->xy, c->cell_vertices, P.grid, cnt, nullptr, nullptr);
    NSG_LAUNCH_CHECK(c);
  }
  const int64_t n_seg = (nb + PT_SCAN_SEG - 1) / PT_SCAN_SEG;
  int64_t *seg = nullptr;
  NSG_TRY(dev_alloc(&seg, n_seg));
  NSG_TRY(dev_alloc(&P.start, nb + 1));
  k_pt_scan_sums<<<(unsigned)n_seg, PT_SCAN_THREADS, 0, c->stream>>>(nb, cnt, seg);
  NSG_LAUNCH_CHECK(c);
  k_pt_scan_top<<<1, PT_SCAN_THREADS, 0, c->stream>>>(n_seg, seg);
  NSG_LAUNCH_CHECK(c);
  k_pt_scan_apply<<<(unsigned)n_seg, PT_SCAN_THREADS, 0, c->stream>>>(nb, cnt, seg, P.start);
  NSG_LAUNCH_CHECK(c);
  // occupancy statistics from the counts (before they become cursors)
  unsigned long long *stats = nullptr, h_stats[2];
  NSG_TRY(dev_alloc(&stats, 2));
  NSG_CUDA(cudaMemsetAsync(stats, 0, 16, c->stream));
  k_pt_bin_stats<<<grid_for(nb, 256), 256, 0, c->stream>>>(nb, cnt, stats);
  NSG_LAUNCH_CHECK(c);
  NSG_CUDA(cudaMemcpyAsync(h_stats, stats, 16, cudaMemcpyDeviceToHost, c->stream));
  NSG_CUDA(cudaMemcpyAsync(&P.n_entries, P.start + nb, 8, cudaMemcpyDeviceToHost, c->stream));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  dev_free(stats);
  P.n_nonempty = (int64_t)h_stats[0], P.max_bin = (int32_t)h_stats[1];
  NSG_TRY(dev_alloc(&P.entries, P.n_entries));
  NSG_CUDA(cudaMemsetAsync(cnt, 0, 4 * (size_t)nb, c->stream));
  if (T > 0) {
    k_pt_bin_cells<1><<<grid, 256, 0, c->stream>>>(T, c->xy, c->cell_vertices, P.grid, cnt, P.start, P.entries);
    NSG_LAUNCH_CHECK(c);
  }
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  dev_free(cnt), dev_free(seg);
  P.built = true;
  P.build_ms = 1e3 * (omp_get_wtime() - t0);
  return NSG_OK;
}

static int pt_ensure_scratch(nsg_ctx *c, int64_t n, bool grads) {
  PointIndex &P = c->pidx;
  if (n > P.cap) {
    dev_free(P.pxy), dev_free(P.vals), dev_free(P.grads), dev_free(P.gid), dev_free(P.win), dev_free(P.loc), dev_free(P.cell);
    P.cap = P.grads_cap = 0;
    NSG_TRY(dev_alloc(&P.pxy, 2 * n));
    NSG_TRY(dev_alloc(&P.vals, 3 * n));
    NSG_TRY(dev_alloc(&P.gid, n));
    NSG_TRY(dev_alloc(&P.win, n));
    NSG_TRY(dev_alloc(&P.loc, n));
    NSG_TRY(dev_alloc(&P.cell, n));
    P.cap = n;
  }
  if (grads && n > P.grads_cap) {
    dev_free(P.grads);
    NSG_TRY(dev_alloc(&P.grads, 6 * P.cap));
    P.grads_cap = P.cap;
  }
  return NSG_OK;
}

// locate + evaluate the n points in P.pxy; collective: combine over the communicator (min of the global id, then sum)
static int pt_run(nsg_ctx *c, int64_t n, bool collective, bool grads) {
  PointIndex &P = c->pidx;
  const int grid = grid_for(n, 128);
  k_pt_locate<<<grid, 128, 0, c->stream>>>(n, P.pxy, P.grid, P.start, P.entries, c->xy, c->cell_vertices, c->geom8, c->cell_gid,
                                          c->cell_owned, P.gid, P.loc);
  NSG_LAUNCH_CHECK(c);
  const int32_t *win = P.gid;
  if (collective) {
    NSG_NCCL(nccl_api().AllReduce(P.gid, P.win, (size_t)n, ncclInt32, ncclMin, c->comm, c->stream));
    win = P.win;
  }
  k_pt_eval<<<grid, 128, 0, c->stream>>>(n, P.pxy, P.gid, P.loc, win, c->xy, c->cell_vertices, c->geom8, c->cell_dofs, c->sol, P.vals,
                                        grads ? P.grads : nullptr, P.cell);
  NSG_LAUNCH_CHECK(c);
  if (collective) {
    NSG_NCCL(nccl_api().AllReduce(P.vals, P.vals, 3 * (size_t)n, ncclDouble, ncclSum, c->comm, c->stream));
    if (grads) NSG_NCCL(nccl_api().AllReduce(P.grads, P.grads, 6 * (size_t)n, ncclDouble, ncclSum, c->comm, c->stream));
  }
  return NSG_OK;
}

static void pt_free(nsg_ctx *c) {
  PointIndex &P = c->pidx;
  dev_free(P.start), dev_free(P.entries);
  dev_free(P.pxy), dev_free(P.vals), dev_free(P.grads), dev_free(P.gid), dev_free(P.win), dev_free(P.loc), dev_free(P.cell);
  dev_free(c->cell_gid), dev_free(c->cell_owned);
}

}  // namespace nsg
