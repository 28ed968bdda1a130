// nsg.cu — libnsg.so: C-ABI of include/nsg.h over the CUDA kernels in nsg_assemble.cuh,
// nsg_linalg.cuh and nsg_precond.cuh (sm_100a, fp64).  One context = one GPU = one rank.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <numeric>
#include <omp.h>

#include "nsg_assemble.cuh"
#include "nsg_assemble_fan.cuh"
#include "nsg_pattern.cuh"
#include "nsg_common.cuh"
#include "nsg_linalg.cuh"

namespace nsg {
thread_local std::string g_err;
int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}

// NSG_TRACE=1: wall-clock marks of the one-time setup calls on stderr
struct Trace {
  bool on;
  double t0;
  const char *what;
  explicit Trace(const char *w) : on(std::getenv("NSG_TRACE") != nullptr), t0(0), what(w) {
    if (on) t0 = omp_get_wtime();
  }
  void mark(const char *label) {
    if (!on) return;
    const double t = omp_get_wtime();
    std::fprintf(stderr, "[nsg trace] %s: %s %.3f s\n", what, label, t - t0);
    t0 = t;
  }
};

template <class T>
int dev_alloc(T **p, int64_t n) {
  *p = nullptr;
  NSG_CUDA(cudaMalloc((void **)p, sizeof(T) * (size_t)std::max<int64_t>(n, 1)));
  return NSG_OK;
}
template <class T>
int upload(nsg_ctx *c, T **p, const T *h, int64_t n) {
  NSG_TRY(dev_alloc(p, n));
  if (n > 0) NSG_CUDA(cudaMemcpyAsync(*p, h, sizeof(T) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  c->h2d += (int64_t)sizeof(T) * n;
  return NSG_OK;
}
template <class T>
void dev_free(T *&p) {
  if (p) cudaFree(p);
  p = nullptr;
}

// number of SMs of the current device (148 on a B200; a MIG/MPS slice has fewer): every persistent grid is sized from it
inline int sm_count() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}
inline int grid_for(int64_t n, int threads, int cap = 0) {
  if (cap <= 0) cap = sm_count() * 16;
  return (int)std::max<int64_t>(1, std::min<int64_t>((n + threads - 1) / threads, cap));
}
inline int red_grid(int64_t n) {
  return (int)std::max<int64_t>(1, std::min<int64_t>(((n >> 1) + RED_THREADS * 4 - 1) / (RED_THREADS * 4), RED_MAX_BLOCKS));
}

// -------------------------------------------------------------------------------------------------
// reference-cell tables
// -------------------------------------------------------------------------------------------------
static void p2_eval(double x, double y, double psi[6], double dpsi[6][2]) {
  const double l0 = 1 - x - y, l1 = x, l2 = y;
  psi[0] = l0 * (2 * l0 - 1), psi[1] = l1 * (2 * l1 - 1), psi[2] = l2 * (2 * l2 - 1);
  psi[3] = 4 * l0 * l1, psi[4] = 4 * l1 * l2, psi[5] = 4 * l2 * l0;
  const double d[3][2] = {{-1, -1}, {1, 0}, {0, 1}};
  for (int c = 0; c < 2; ++c) {
    dpsi[0][c] = (4 * l0 - 1) * d[0][c];
    dpsi[1][c] = (4 * l1 - 1) * d[1][c];
    dpsi[2][c] = (4 * l2 - 1) * d[2][c];
    dpsi[3][c] = 4 * (l0 * d[1][c] + l1 * d[0][c]);
    dpsi[4][c] = 4 * (l1 * d[2][c] + l2 * d[1][c]);
    dpsi[5][c] = 4 * (l2 * d[0][c] + l0 * d[2][c]);
  }
}
static int upload_tables() {
  FeTables t;
  const double s = std::sqrt(15.0);
  const double a = (6.0 - s) / 21.0, b = (6.0 + s) / 21.0;
  const double wa = (155.0 - s) / 2400.0, wb = (155.0 + s) / 2400.0;
  const double px[7] = {1.0 / 3.0, 1 - 2 * a, a, a, 1 - 2 * b, b, b};
  const double py[7] = {1.0 / 3.0, a, 1 - 2 * a, a, b, 1 - 2 * b, b};
  const double pw[7] = {9.0 / 80.0, wa, wa, wa, wb, wb, wb};
  for (int q = 0; q < 7; ++q) {
    t.w[q] = pw[q];
    p2_eval(px[q], py[q], t.psi[q], t.dpsi[q]);
    t.chi[q][0] = 1 - px[q] - py[q], t.chi[q][1] = px[q], t.chi[q][2] = py[q];
  }
  for (int k = 0; k < 6; ++k)
    for (int l = 0; l < 6; ++l) {
      double m = 0;
      for (int q = 0; q < 7; ++q) m += t.w[q] * t.psi[q][k] * t.psi[q][l];
      t.mhat[k][l] = m;
    }
  t.gl[0] = 0.5 - 0.5 * std::sqrt(0.6), t.gl[1] = 0.5, t.gl[2] = 0.5 + 0.5 * std::sqrt(0.6);
  t.gw[0] = 5.0 / 18.0, t.gw[1] = 8.0 / 18.0, t.gw[2] = 5.0 / 18.0;
  NSG_CUDA(cudaMemcpyToSymbol(c_fe, &t, sizeof t));
  // pre-integrated tables of the factored kernels, from the same rule
  FeTables2 f;
  std::memset(&f, 0, sizeof f);
  for (int q = 0; q < 7; ++q) {
    f.qx[q] = px[q], f.qy[q] = py[q];
    for (int k = 0; k < 6; ++k) {
      f.mh[k] += t.w[q] * t.psi[q][k];
      for (int l = 0; l < 6; ++l) {
        const double m = t.w[q] * t.psi[q][k] * t.psi[q][l];
        f.Mh[k][l] += m;
        f.Mx[k][l] += m * px[q];
        f.My[k][l] += m * py[q];
        f.K00[k][l] += t.w[q] * t.dpsi[q][k][0] * t.dpsi[q][l][0];
        f.K01s[k][l] += t.w[q] * (t.dpsi[q][k][0] * t.dpsi[q][l][1] + t.dpsi[q][k][1] * t.dpsi[q][l][0]);
        f.K11[k][l] += t.w[q] * t.dpsi[q][k][1] * t.dpsi[q][l][1];
      }
      for (int m = 0; m < 3; ++m)
        for (int c = 0; c < 2; ++c) f.Bh[k][m][c] += t.w[q] * t.dpsi[q][k][c] * t.chi[q][m];
    }
    for (int m = 0; m < 3; ++m)
      for (int n = 0; n < 3; ++n) f.Mp[m][n] += t.w[q] * t.chi[q][m] * t.chi[q][n];
  }
  {
    double p0[6], g0[6][2], gx[6][2], gy[6][2];
    p2_eval(0, 0, p0, g0);
    p2_eval(1, 0, p0, gx);
    p2_eval(0, 1, p0, gy);
    for (int l = 0; l < 6; ++l)
      for (int c = 0; c < 2; ++c) f.ga[l][c] = g0[l][c], f.gb[l][c] = gx[l][c] - g0[l][c], f.gc[l][c] = gy[l][c] - g0[l][c];
  }
  NSG_CUDA(cudaMemcpyToSymbol(c_fe2, &f, sizeof f));
  // rows of the tables for the owner's local index in the rotated frame of the fan scheme (K = 0 vertex, K = 3 edge midpoint)
  FanTab ft[2];
  std::memset(ft, 0, sizeof ft);
  for (int i = 0; i < 2; ++i) {
    const int K = i == 0 ? 0 : 3;
    for (int q = 0; q < 7; ++q)
      for (int l = 0; l < 6; ++l) {
        const double m = t.w[q] * t.psi[q][K] * t.psi[q][l];
        ft[i].M[l] += m;
        for (int j = 0; j < 3; ++j) ft[i].T[j][l] += m * t.chi[q][j];
        ft[i].K00[l] += t.w[q] * t.dpsi[q][K][0] * t.dpsi[q][l][0];
        ft[i].K01s[l] += t.w[q] * (t.dpsi[q][K][0] * t.dpsi[q][l][1] + t.dpsi[q][K][1] * t.dpsi[q][l][0]);
        ft[i].K11[l] += t.w[q] * t.dpsi[q][K][1] * t.dpsi[q][l][1];
      }
    for (int m = 0; m < 3; ++m)
      for (int cc = 0; cc < 2; ++cc) ft[i].Bh[m][cc] = f.Bh[K][m][cc];
  }
  NSG_CUDA(cudaMemcpyToSymbol(c_fan, ft, sizeof ft));
  FanTabP fp;
  for (int l = 0; l < 6; ++l)
    for (int cc = 0; cc < 2; ++cc) fp.Bp[l][cc] = f.Bh[l][0][cc];
  for (int n = 0; n < 3; ++n) fp.Mp[n] = f.Mp[0][n];
  NSG_CUDA(cudaMemcpyToSymbol(c_fanp, &fp, sizeof fp));
  return NSG_OK;
}

// -------------------------------------------------------------------------------------------------
// row-owner work lists (host, once)
// -------------------------------------------------------------------------------------------------
// Cells per row owner (= vertex valence) each assembly variant serves: variant 0 puts an owner's pairs two per lane into
// one warp, variant 4 one per lane (the 5-bit commit round of its record holds 0..31), the fan scheme (variant 5,
// nsg_fanlist.inl) one per lane.
constexpr int ASM_MAX_VALENCE_0 = 64, ASM_MAX_VALENCE_4 = 32, ASM_MAX_VALENCE_5 = 32;

// the largest number of cells of one owned row owner (velocity node or pressure vertex)
static int max_owner_cells(const nsg_ctx *c, const int32_t *cd) {
  const int64_t nu = c->n_own_u, nown = c->n_own;
  std::vector<int32_t> cnt((size_t)(nu / 2 + c->n_own_p), 0);
  for (int64_t cell = 0; cell < c->n_cells; ++cell)
    for (int k = 0; k < 9; ++k) {
      const int32_t d = cd[15 * cell + (k < 6 ? uidx(k) : 3 * (k - 6) + 2)];
      if (d < nu) cnt[(size_t)(d / 2)]++;
      else if (d < nown) cnt[(size_t)(nu / 2 + d - nu)]++;
    }
  return cnt.empty() ? 0 : *std::max_element(cnt.begin(), cnt.end());
}

static int build_worklist(nsg_ctx *c, int kind, const int32_t *cd, WorkList *out) {
  const int64_t T = c->n_cells, nu = c->n_own_u, nown = c->n_own;
  const int64_t ng = kind == 0 ? nu / 2 : c->n_own_p;
  const int nk = kind == 0 ? 6 : 3;
  auto group_of = [&](int64_t cell, int k) -> int64_t {
    const int32_t d = cd[15 * cell + (kind == 0 ? uidx(k) : 3 * k + 2)];
    if (kind == 0) return d < nu ? d / 2 : -1;
    return (d >= nu && d < nown) ? d - nu : -1;
  };
  std::vector<int64_t> gptr(ng + 1, 0);
  for (int64_t cell = 0; cell < T; ++cell)
    for (int k = 0; k < nk; ++k) {
      const int64_t g = group_of(cell, k);
      if (g >= 0) gptr[g + 1]++;
    }
  for (int64_t g = 0; g < ng; ++g) gptr[g + 1] += gptr[g];
  const int64_t npairs = gptr[ng];
  std::vector<int32_t> pcell(npairs);
  std::vector<uint8_t> pk(npairs);
  {
    std::vector<int64_t> pos(gptr.begin(), gptr.end() - 1);
    for (int64_t cell = 0; cell < T; ++cell)
      for (int k = 0; k < nk; ++k) {
        const int64_t g = group_of(cell, k);
        if (g >= 0) {
          pcell[pos[g]] = (int32_t)cell;
          pk[pos[g]++] = (uint8_t)k;
        }
      }
  }
  // chunks: consecutive owners while their slots fit one CTA.  The slots of one owner occupy adjacent
  // lanes of ONE warp (an owner never straddles a warp: pad to the next warp instead), so the ordered
  // commit of an owner's pairs needs only __syncwarp(), never a CTA barrier.
  auto nslots = [&](int64_t g) { return std::max((int)((gptr[g + 1] - gptr[g] + ASM_PPT - 1) / ASM_PPT), 1); };
  // staged entries (shared-memory image) of owner g; a cap on the image keeps more CTAs resident per SM
  auto stage_of = [&](int64_t g) -> int64_t {
    if (kind == 0) return c->h_rowptr[2 * g + 2] - c->h_rowptr[2 * g] + 2;
    return (c->h_rowptr[nu + g + 1] - c->h_rowptr[nu + g]) + (c->h_pm_rowptr[nu + g + 1] - c->h_pm_rowptr[nu + g]);
  };
  const int64_t stage_cap = std::getenv("NSG_ASM_STAGE_CAP") ? std::atoll(std::getenv("NSG_ASM_STAGE_CAP")) : ASM_STAGE_CAP;
  std::vector<ChunkInfo> chunks;
  {
    int64_t g = 0, rec = 0;
    while (g < ng) {
      ChunkInfo ci{};
      ci.g0 = (int32_t)g;
      int nt = 0, mx = 0;
      int64_t staged = 0;
      while (g < ng && g - ci.g0 < 255) {
        const int ns = nslots(g);
        if (gptr[g + 1] - gptr[g] > ASM_MAX_VALENCE_0)
          return fail(NSG_ERR_ARG, "a vertex has " + std::to_string(gptr[g + 1] - gptr[g]) + " incident cells: assembly variant 0 serves at most " +
                                       std::to_string(ASM_MAX_VALENCE_0));
        int pos = nt;
        if ((pos & 31) + ns > 32) pos = (pos + 31) & ~31;  // next warp
        if (pos + ns > NPC) break;
        if (g > ci.g0 && staged + stage_of(g) > stage_cap) break;
        staged += stage_of(g);
        nt = pos + ns;
        mx = std::max(mx, ns);
        ++g;
      }
      ci.g1 = (int32_t)g;
      ci.n_threads = nt;
      ci.max_slots = mx;
      ci.rec_base = rec;
      if (kind == 0) {
        ci.rs = c->h_rowptr[2 * (int64_t)ci.g0];
        ci.cnt = (int32_t)(c->h_rowptr[2 * (int64_t)ci.g1] - ci.rs);
      } else {
        ci.rs = c->h_rowptr[nu + ci.g0], ci.ms = c->h_pm_rowptr[nu + ci.g0];
        ci.cnt = (int32_t)(c->h_rowptr[nu + ci.g1] - ci.rs), ci.mcnt = (int32_t)(c->h_pm_rowptr[nu + ci.g1] - ci.ms);
      }
      rec += (int64_t)nt * ASM_PPT;
      chunks.push_back(ci);
    }
  }
  const int64_t nchunks = (int64_t)chunks.size();
  const int64_t nrecs = nchunks ? chunks.back().rec_base + (int64_t)chunks.back().n_threads * ASM_PPT : 0;
  std::vector<uint16_t> tdesc((size_t)nchunks * NPC, 0xffff);  // 0xffff = padding lane
  std::vector<uint2> tdesc3((size_t)nchunks * NPC, make_uint2(0u, 0xffffffffu));
  std::vector<PairRec> recs(nrecs);
  int bad = 0;
  int64_t max_stage = 0;
#pragma omp parallel for schedule(dynamic, 64) reduction(max : max_stage) reduction(+ : bad)
  for (int64_t b = 0; b < nchunks; ++b) {
    const ChunkInfo &ci = chunks[b];
    PairRec empty;
    std::memset(&empty, 0, sizeof empty);
    empty.cell = -1;
    for (int j = 0; j < ASM_PPT; ++j)
      for (int t = 0; t < ci.n_threads; ++t) recs[ci.rec_base + (int64_t)j * ci.n_threads + t] = empty;
    int t = 0;
    for (int64_t g = ci.g0; g < ci.g1; ++g) {
      const int ns = nslots(g);
      if ((t & 31) + ns > 32) t = (t + 31) & ~31;
      for (int r = 0; r < ns; ++r, ++t) {
        tdesc[b * NPC + t] = (uint16_t)((g - ci.g0) | (r << 8));
        {
          const int64_t row = kind == 0 ? 2 * g : nu + g;
          const int64_t off = c->h_rowptr[row] - ci.rs, len = c->h_rowptr[row + 1] - c->h_rowptr[row];
          const int64_t moff = kind == 0 ? 0 : c->h_pm_rowptr[row] - ci.ms;
          if (off >= 65536 || moff >= 65536 || len >= 65536) bad++;
          tdesc3[b * NPC + t] = make_uint2((uint32_t)(off | (moff << 16)), (uint32_t)(len | ((uint32_t)r << 16) | ((uint32_t)(g - ci.g0) << 24)));
        }
        for (int j = 0; j < ASM_PPT; ++j) {
          const int64_t pi = r + (int64_t)j * ns;
          if (pi >= gptr[g + 1] - gptr[g]) continue;
          PairRec rcd = empty;
          const int64_t src = gptr[g] + pi;
          rcd.cell = pcell[src];
          rcd.k = pk[src];
          const int32_t *cdc = cd + 15 * (int64_t)rcd.cell;
          const int64_t row = kind == 0 ? 2 * g : nu + g;
          const int64_t rs = c->h_rowptr[row], re = c->h_rowptr[row + 1];
          if (re - rs >= 65535) bad++;
          if (kind == 0 && c->h_rowptr[row + 2] - re != re - rs) bad++;
          const int32_t *cb = c->h_col.data() + rs, *ce = c->h_col.data() + re;
          for (int l = 0; l < 6; ++l) {
            const int32_t tgt = cdc[uidx(l)];
            const int32_t *p = std::lower_bound(cb, ce, tgt);
            if (p == ce || *p != tgt || p + 1 == ce || p[1] != tgt + 1) {
              bad++;
              continue;
            }
            rcd.off[l] = (uint16_t)(p - cb);
          }
          const int32_t *mb = cb, *me = ce;
          if (kind == 1) {
            mb = c->h_pm_col.data() + c->h_pm_rowptr[row];
            me = c->h_pm_col.data() + c->h_pm_rowptr[row + 1];
          }
          for (int m = 0; m < 3; ++m) {
            const int32_t tgt = cdc[3 * m + 2];
            const int32_t *p = std::lower_bound(mb, me, tgt);
            if (p == me || *p != tgt) {
              bad++;
              continue;
            }
            rcd.off[6 + m] = (uint16_t)(p - mb);
          }
          recs[ci.rec_base + (int64_t)j * ci.n_threads + t] = rcd;
        }
      }
    }
    if (t != ci.n_threads) bad++;
    int64_t stage;
    if (kind == 0)
      stage = c->h_rowptr[2 * (int64_t)ci.g1] - c->h_rowptr[2 * (int64_t)ci.g0] + 2 * (ci.g1 - ci.g0);
    else
      stage = (c->h_rowptr[nu + ci.g1] - c->h_rowptr[nu + ci.g0]) + (c->h_pm_rowptr[nu + ci.g1] - c->h_pm_rowptr[nu + ci.g0]);
    max_stage = std::max(max_stage, stage);
  }
  if (bad) return fail(NSG_ERR_ARG, "cell_dofs do not match the sparsity pattern (or a row has >= 65535 entries)");
  out->n_groups = ng;
  out->n_chunks = nchunks;
  out->n_pairs = npairs;
  out->n_recs = nrecs;
  out->max_stage = max_stage + 2;  // the 128-bit zero-fill may touch one padding element
  NSG_TRY(upload(c, &out->chunks, chunks.data(), nchunks));
  NSG_TRY(upload(c, &out->tdesc, tdesc.data(), (int64_t)tdesc.size()));
  NSG_TRY(upload(c, &out->tdesc3, tdesc3.data(), (int64_t)tdesc3.size()));
  NSG_TRY(upload(c, &out->recs, recs.data(), nrecs));
  NSG_CUDA(cudaStreamSynchronize(c->stream));  // host vectors die here
  return NSG_OK;
}

// Work list of assembly variant 4 (k_assemble_u5 / k_assemble_p5): ONE (owner, cell) pair per lane, the lanes
// of a chunk sorted by (commit round, cell).  Round = rank of the cell among the owner's cells, so all lanes
// of a warp commit together (full shared-memory wavefronts instead of 3 mostly idle rounds per warp) and
// lanes that read the same cell packet sit next to each other (fewer L1 wavefronts per load).  The record
// carries everything the lane needs: no descriptor array, no row-pointer loads.
//   rec.k    = k | round << 3 | owner-in-chunk << 8 | first-touch bits of the 9 column groups << 16 | first-touch of R << 25
//   rec.off  = [0..8] column offsets (as PairRec), [9] image offset of the owner's first row (pressure: J row),
//              [10] row length (pressure: image offset of the pressure-mass row)
static int build_worklist5(nsg_ctx *c, int kind, const int32_t *cd, WorkList *out) {
  const int64_t T = c->n_cells, nu = c->n_own_u, nown = c->n_own;
  const int64_t ng = kind == 0 ? nu / 2 : c->n_own_p;
  const int nk = kind == 0 ? 6 : 3;
  auto group_of = [&](int64_t cell, int k) -> int64_t {
    const int32_t d = cd[15 * cell + (kind == 0 ? uidx(k) : 3 * k + 2)];
    if (kind == 0) return d < nu ? d / 2 : -1;
    return (d >= nu && d < nown) ? d - nu : -1;
  };
  std::vector<int64_t> gptr(ng + 1, 0);
  for (int64_t cell = 0; cell < T; ++cell)
    for (int k = 0; k < nk; ++k) {
      const int64_t g = group_of(cell, k);
      if (g >= 0) gptr[g + 1]++;
    }
  for (int64_t g = 0; g < ng; ++g) gptr[g + 1] += gptr[g];
  const int64_t npairs = gptr[ng];
  std::vector<int32_t> pcell(npairs);
  std::vector<uint8_t> pk(npairs);
  {
    std::vector<int64_t> pos(gptr.begin(), gptr.end() - 1);
    for (int64_t cell = 0; cell < T; ++cell)  // ascending cell order per owner
      for (int k = 0; k < nk; ++k) {
        const int64_t g = group_of(cell, k);
        if (g >= 0) {
          pcell[pos[g]] = (int32_t)cell;
          pk[pos[g]++] = (uint8_t)k;
        }
      }
  }
  auto stage_of = [&](int64_t g) -> int64_t {
    if (kind == 0) return c->h_rowptr[2 * g + 2] - c->h_rowptr[2 * g] + 2;
    return (c->h_rowptr[nu + g + 1] - c->h_rowptr[nu + g]) + (c->h_pm_rowptr[nu + g + 1] - c->h_pm_rowptr[nu + g]);
  };
  const int64_t stage_cap = std::getenv("NSG_ASM_STAGE_CAP") ? std::atoll(std::getenv("NSG_ASM_STAGE_CAP")) : ASM_STAGE_CAP;
  std::vector<ChunkInfo> chunks;
  {
    int64_t g = 0, rec = 0;
    while (g < ng) {
      ChunkInfo ci{};
      ci.g0 = (int32_t)g;
      int nt = 0, mx = 0;
      int64_t staged = 0;
      while (g < ng && g - ci.g0 < 255) {
        const int np = (int)(gptr[g + 1] - gptr[g]);
        if (np > ASM_MAX_VALENCE_4)
          return fail(NSG_ERR_ARG, "a vertex has " + std::to_string(np) + " incident cells: assembly variant 4 serves at most " +
                                       std::to_string(ASM_MAX_VALENCE_4));
        if (nt + np > NPC5 && g > ci.g0) break;
        if (g > ci.g0 && staged + stage_of(g) > stage_cap) break;
        staged += stage_of(g);
        nt += np;
        mx = std::max(mx, np);
        ++g;
      }
      ci.g1 = (int32_t)g;
      ci.n_threads = nt;
      ci.max_slots = mx;
      ci.rec_base = rec;  // == chunk index * NPC5: a lane finds its record without reading the chunk header
      if (kind == 0) {
        ci.rs = c->h_rowptr[2 * (int64_t)ci.g0];
        ci.cnt = (int32_t)(c->h_rowptr[2 * (int64_t)ci.g1] - ci.rs);
      } else {
        ci.rs = c->h_rowptr[nu + ci.g0], ci.ms = c->h_pm_rowptr[nu + ci.g0];
        ci.cnt = (int32_t)(c->h_rowptr[nu + ci.g1] - ci.rs), ci.mcnt = (int32_t)(c->h_pm_rowptr[nu + ci.g1] - ci.ms);
      }
      rec += NPC5;
      chunks.push_back(ci);
    }
  }
  const int64_t nchunks = (int64_t)chunks.size();
  PairRec no_work;
  std::memset(&no_work, 0, sizeof no_work);
  no_work.cell = -1;
  std::vector<PairRec> recs((size_t)nchunks * NPC5, no_work);
  int bad = 0;
  int64_t max_stage = 0;
#pragma omp parallel for schedule(dynamic, 64) reduction(max : max_stage) reduction(+ : bad)
  for (int64_t b = 0; b < nchunks; ++b) {
    ChunkInfo &ci = chunks[b];
    struct Lane {
      int32_t round, cell, k, gl;
    };
    std::vector<Lane> lanes;
    lanes.reserve(NPC5);
    for (int64_t g = ci.g0; g < ci.g1; ++g)
      for (int64_t pi = gptr[g]; pi < gptr[g + 1]; ++pi) lanes.push_back({(int32_t)(pi - gptr[g]), pcell[pi], pk[pi], (int32_t)(g - ci.g0)});
    std::sort(lanes.begin(), lanes.end(), [](const Lane &a, const Lane &b2) {
      if (a.round != b2.round) return a.round < b2.round;
      if (a.cell != b2.cell) return a.cell < b2.cell;
      return a.k < b2.k;
    });
    if ((int)lanes.size() != ci.n_threads || ci.n_threads > NPC5) bad++;
    // first-touch bookkeeping per image entry
    const int64_t img = kind == 0 ? ci.cnt : (int64_t)ci.cnt + ci.mcnt;
    std::vector<uint8_t> touched((size_t)img, 0), rtouched((size_t)(ci.g1 - ci.g0), 0);
    int64_t n_touched = 0;
    for (size_t t = 0; t < lanes.size(); ++t) {
      const Lane &ln = lanes[t];
      PairRec rcd;
      std::memset(&rcd, 0, sizeof rcd);
      rcd.cell = ln.cell;
      const int64_t g = ci.g0 + ln.gl;
      const int32_t *cdc = cd + 15 * (int64_t)ln.cell;
      const int64_t row = kind == 0 ? 2 * g : nu + g;
      const int64_t rs = c->h_rowptr[row], re = c->h_rowptr[row + 1];
      const int64_t len = re - rs, roff = rs - ci.rs;
      if (len >= 65535 || roff >= 65535) bad++;
      if (kind == 0 && c->h_rowptr[row + 2] - re != len) bad++;
      uint32_t first = 0;
      const int32_t *cb = c->h_col.data() + rs, *ce = c->h_col.data() + re;
      for (int l = 0; l < 6; ++l) {
        const int32_t tgt = cdc[uidx(l)];
        const int32_t *p = std::lower_bound(cb, ce, tgt);
        if (p == ce || *p != tgt || p + 1 == ce || p[1] != tgt + 1) {
          bad++;
          continue;
        }
        rcd.off[l] = (uint16_t)(p - cb);
        // lanes are visited in commit order (round-major), so "not yet touched" == first contribution
        uint8_t &f = touched[(size_t)(roff + (p - cb))];
        if (!f) {
          first |= 1u << l;
          f = 1;
          n_touched += kind == 0 ? 4 : 2;
          touched[(size_t)(roff + (p - cb) + 1)] = 1;
          if (kind == 0) touched[(size_t)(roff + len + (p - cb))] = touched[(size_t)(roff + len + (p - cb) + 1)] = 1;
        }
      }
      const int32_t *mb = cb, *me = ce;
      int64_t moff = roff;
      if (kind == 1) {
        mb = c->h_pm_col.data() + c->h_pm_rowptr[row];
        me = c->h_pm_col.data() + c->h_pm_rowptr[row + 1];
        moff = ci.cnt + (c->h_pm_rowptr[row] - ci.ms);
        if (c->h_pm_rowptr[row] - ci.ms >= 65535) bad++;
      }
      for (int m = 0; m < 3; ++m) {
        const int32_t tgt = cdc[3 * m + 2];
        const int32_t *p = std::lower_bound(mb, me, tgt);
        if (p == me || *p != tgt) {
          bad++;
          continue;
        }
        rcd.off[6 + m] = (uint16_t)(p - mb);
        uint8_t &f = touched[(size_t)(moff + (p - mb))];
        if (!f) {
          first |= 1u << (6 + m);
          f = 1;
          n_touched += 1;
          if (kind == 0) touched[(size_t)(roff + len + (p - mb))] = 1, n_touched += 1;
        }
      }
      uint32_t rfirst = 0;
      if (!rtouched[ln.gl]) rfirst = 1, rtouched[ln.gl] = 1;
      rcd.k = (int32_t)((uint32_t)ln.k | ((uint32_t)ln.round << 3) | ((uint32_t)ln.gl << 8) | (first << 16) | (rfirst << 25));
      rcd.off[9] = (uint16_t)roff;
      rcd.off[10] = kind == 0 ? (uint16_t)len : (uint16_t)(c->h_pm_rowptr[row] - ci.ms);
      recs[ci.rec_base + (int64_t)t] = rcd;
    }
    // an entry of the pattern no cell contributes to (a pattern wider than the mesh implies) must still be written: zero-fill
    bool all_r = true;
    for (uint8_t f : rtouched) all_r &= f != 0;
    ci.pad = (n_touched == img && all_r) ? 0 : 1;
    const int64_t stage = kind == 0 ? (int64_t)ci.cnt + 2 * (ci.g1 - ci.g0) : (int64_t)ci.cnt + ci.mcnt;
    max_stage = std::max(max_stage, stage);
  }
  if (bad) return fail(NSG_ERR_ARG, "cell_dofs do not match the sparsity pattern (or a row has >= 65535 entries)");
  out->n_groups = ng;
  out->n_chunks = nchunks;
  out->n_pairs = npairs;
  out->n_recs = nchunks * NPC5;
  out->max_stage = max_stage + 2;
  NSG_TRY(upload(c, &out->chunks, chunks.data(), nchunks));
  NSG_TRY(upload(c, &out->recs, recs.data(), nchunks * NPC5));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  return NSG_OK;
}

#include "nsg_fanlist.inl"

static void free_worklist(WorkList &w) {
  dev_free(w.chunks);
  dev_free(w.tdesc);
  dev_free(w.tdesc3);
  dev_free(w.recs);
}

// chunks of consecutive rows with <= SPMV_CAP non-zeros and <= SPMV_THREADS rows
static void make_spmv_chunks(const int64_t *rowptr, int64_t n, std::vector<int32_t> &chunks) {
  chunks.clear();
  chunks.push_back(0);
  int64_t r = 0;
  while (r < n) {
    int64_t e = r + 1;
    while (e < n && e - r < SPMV_THREADS && rowptr[e + 1] - rowptr[r] <= SPMV_CAP) ++e;
    chunks.push_back((int32_t)e);
    r = e;
  }
}

// SpMV variant 7 serves the two rows of a velocity node together: true if rows 2g and 2g+1 have the same column list
// for every owned velocity node (full coupling of the two components, cpp:107-110)
static bool rows_come_in_pairs(const nsg_ctx *c, const int64_t *rowptr, const int32_t *col) {
  const int64_t n_ug = c->n_own_u / 2;
  if (c->n_own_u % 2) return false;
  int bad = 0;
#pragma omp parallel for schedule(static) reduction(+ : bad)
  for (int64_t g = 0; g < n_ug; ++g) {
    const int64_t s = rowptr[2 * g], e = rowptr[2 * g + 1];
    if (rowptr[2 * g + 2] - e != e - s || std::memcmp(col + s, col + e, 4 * (size_t)(e - s)) != 0) bad++;
  }
  return bad == 0;
}

// -------------------------------------------------------------------------------------------------
// communication helpers
// -------------------------------------------------------------------------------------------------
// Ghost import, first half: make my owned values visible to the neighbours that hold them as ghosts.  With the peer
// mailboxes mapped (nsg_comm_set_peers) this is ONE kernel storing {value, stamp} words straight into the neighbours'
// inboxes over NVLink; otherwise gather + grouped ncclSend/ncclRecv (which also completes the import).
static int halo_begin(nsg_ctx *c, double *vec) {
  if (c->n_ranks <= 1 || c->n_neighbors == 0) return NSG_OK;
  if (c->halo_peer) {
    if (c->n_send > 0) {
      k_halo_push<<<grid_for(c->n_send, 256, sm_count()), 256, 0, c->stream>>>(c->n_send, c->send_idx, vec, c->send_dst, c->halo_ctr,
                                                                              c->halo_ticket);
      NSG_LAUNCH_CHECK(c);
    }
    return NSG_OK;
  }
  if (c->n_send > 0) {
    k_gather<<<grid_for(c->n_send, 256, 1 << 20), 256, 0, c->stream>>>(c->n_send, c->send_idx, vec, c->send_buf);
    NSG_LAUNCH_CHECK(c);
  }
  NSG_NCCL(nccl_api().GroupStart());
  for (int k = 0; k < c->n_neighbors; ++k) {
    const int64_t ns = c->send_ptr[k + 1] - c->send_ptr[k], nr = c->recv_ptr[k + 1] - c->recv_ptr[k];
    if (ns > 0) NSG_NCCL(nccl_api().Send(c->send_buf + c->send_ptr[k], (size_t)ns, ncclDouble, c->neighbors[k], c->comm, c->stream));
    if (nr > 0) NSG_NCCL(nccl_api().Recv(c->recv_buf + c->recv_ptr[k], (size_t)nr, ncclDouble, c->neighbors[k], c->comm, c->stream));
  }
  NSG_NCCL(nccl_api().GroupEnd());
  if (c->n_recv > 0) {
    k_scatter<<<grid_for(c->n_recv, 256, 1 << 20), 256, 0, c->stream>>>(c->n_recv, c->recv_idx, c->recv_buf, vec);
    NSG_LAUNCH_CHECK(c);
  }
  return NSG_OK;
}
// second half (peer path only): wait for the neighbours' words in my own inbox and write my ghost range
static int halo_end(nsg_ctx *c, double *vec) {
  if (c->n_ranks <= 1 || c->n_neighbors == 0 || !c->halo_peer) return NSG_OK;
  if (c->n_recv > 0) {
    const PeerWord *inbox = reinterpret_cast<const PeerWord *>(c->mailbox + PEER_INBOX_OFFSET);
    k_halo_wait_scatter<<<grid_for(c->n_recv, 256, sm_count()), 256, 0, c->stream>>>(c->n_recv, c->recv_idx, inbox, vec, c->halo_ctr + 1,
                                                                                    c->halo_ticket + 1, c->halo_err);
    NSG_LAUNCH_CHECK(c);
  }
  return NSG_OK;
}
static int halo_exchange(nsg_ctx *c, double *vec) {
  NSG_TRY(halo_begin(c, vec));
  return halo_end(c, vec);
}
static int allreduce_scalar(nsg_ctx *c, double *d) {
  if (c->n_ranks <= 1) return NSG_OK;
  NSG_NCCL(nccl_api().AllReduce(d, d, 1, ncclDouble, ncclSum, c->comm, c->stream));
  return NSG_OK;
}

// -------------------------------------------------------------------------------------------------
// vector-op wrappers (global over ranks)
// -------------------------------------------------------------------------------------------------
// With the peer mailboxes set up (nsg_comm_set_peers) the all-reduce is fused into the reduction kernel;
// otherwise NCCL does it.
static inline bool fused_ar(const nsg_ctx *c) { return c->peer.n_ranks > 1; }
static int dev_dot(nsg_ctx *c, int64_t n, const double *a, const double *b, double *out, const int32_t *state) {
  k_dot<<<red_grid(n), RED_THREADS, 0, c->stream>>>(n, a, b, c->partials, c->ticket, out, state, c->peer);
  NSG_LAUNCH_CHECK(c);
  return fused_ar(c) ? NSG_OK : allreduce_scalar(c, out);
}
static int dev_add_and_dot(nsg_ctx *c, int64_t n, double *vv, const double *aptr, double sign, const double *V,
                           const double *W, double *out, const int32_t *state) {
  k_add_and_dot<<<red_grid(n), RED_THREADS, 0, c->stream>>>(n, vv, aptr, sign, V, W, c->partials, c->ticket, out, state, c->peer);
  NSG_LAUNCH_CHECK(c);
  return fused_ar(c) ? NSG_OK : allreduce_scalar(c, out);
}
// classical Gram-Schmidt building blocks (global over ranks)
static int dev_multi_dot(nsg_ctx *c, int64_t n, const double *w, const double *basis, int k, double *out, const int32_t *state) {
  k_multi_dot<<<red_grid(n), RED_THREADS, 0, c->stream>>>(n, w, basis, c->stride, k, c->partials_k, c->ticket, out, state, c->peer);
  NSG_LAUNCH_CHECK(c);
  if (c->n_ranks > 1 && !fused_ar(c)) NSG_NCCL(nccl_api().AllReduce(out, out, (size_t)k, ncclDouble, ncclSum, c->comm, c->stream));
  return NSG_OK;
}
static int dev_multi_axpy_norm(nsg_ctx *c, int64_t n, double *w, const double *basis, const double *h, int k, double *out,
                               const int32_t *state) {
  k_multi_axpy_norm<<<red_grid(n), RED_THREADS, 0, c->stream>>>(n, w, basis, c->stride, h, k, c->partials, c->ticket, out, state, c->peer);
  NSG_LAUNCH_CHECK(c);
  return fused_ar(c) ? NSG_OK : allreduce_scalar(c, out);
}

static int dev_spmv(nsg_ctx *c, double *x_with_ghosts, double *y, const int32_t *state) {
  if (c->spmv_variant == 7) {
    static int per_sm7 = 0;
    if (!per_sm7) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm7, k_spmv_rowpair<true>, SPMV_THREADS, 0);
    const int64_t n_groups = c->n_own_u / 2 + c->n_own_p;
    // peer-store halo: the sweep over ALL rows runs while the neighbours' values are in flight; the rows with a ghost
    // column (a list made once, O(sqrt(n)) of them) are then recomputed by the same kernel once the ghosts have landed
    const bool overlap = c->halo_peer && c->n_ranks > 1 && c->n_neighbors > 0 && c->bgroups != nullptr;
    if (overlap)
      NSG_TRY(halo_begin(c, x_with_ghosts));
    else
      NSG_TRY(halo_exchange(c, x_with_ghosts));
    k_spmv_rowpair<true><<<(unsigned)std::min<int64_t>((n_groups * 8 + SPMV_THREADS - 1) / SPMV_THREADS, (int64_t)sm_count() * std::max(per_sm7, 1)),
                           SPMV_THREADS, 0, c->stream>>>(c->n_own_u / 2, c->n_own, c->rowptr, c->col, c->vals, x_with_ghosts, y, state);
    if (overlap) {
      NSG_LAUNCH_CHECK(c);
      NSG_TRY(halo_end(c, x_with_ghosts));
      if (c->n_bgroups > 0)
        k_spmv_rowpair_list<<<(unsigned)((c->n_bgroups * 8 + SPMV_THREADS - 1) / SPMV_THREADS), SPMV_THREADS, 0, c->stream>>>(
            c->n_bgroups, c->bgroups, c->n_own_u / 2, c->rowptr, c->col, c->vals, x_with_ghosts, y, state);
    }
    NSG_LAUNCH_CHECK(c);
    return NSG_OK;
  }
  NSG_TRY(halo_exchange(c, x_with_ghosts));
  if (c->spmv_variant == 4) {
    static int per_sm = 0;
    if (!per_sm) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_spmv_vec8u<true>, SPMV_THREADS, 0);
    k_spmv_vec8u<true><<<(unsigned)std::min<int64_t>((c->n_own * 8 + SPMV_THREADS - 1) / SPMV_THREADS, (int64_t)sm_count() * std::max(per_sm, 1)),
                         SPMV_THREADS, 0, c->stream>>>(c->n_own, c->rowptr, c->col, c->vals, x_with_ghosts, y, state);
  } else if (c->spmv_variant == 1)
    k_spmv_vec8<<<(unsigned)((c->n_own * 8 + SPMV_THREADS - 1) / SPMV_THREADS), SPMV_THREADS, 0, c->stream>>>(
        c->n_own, c->rowptr, c->col, c->vals, x_with_ghosts, y, state);
  else
    k_spmv_stream<<<(unsigned)c->spmv_n_chunks, SPMV_THREADS, 0, c->stream>>>(c->spmv_chunk_rows, c->rowptr, c->col, c->vals,
                                                                              x_with_ghosts, y, state);
  NSG_LAUNCH_CHECK(c);
  return NSG_OK;
}

static AsmParams asm_params(const nsg_ctx *c) {
  AsmParams P;
  P.nu = c->prm.nu, P.rho = c->prm.rho, P.p_out = c->prm.p_out;
  P.dt_inv = c->prm.use_mass ? 1.0 / c->prm.deltat : 0.0;
  P.f0 = c->prm.forcing[0], P.f1 = c->prm.forcing[1];
  P.use_mass = c->prm.use_mass, P.stokes = c->prm.stokes, P.neumann_id = c->prm.neumann_id;
  P.debug = std::getenv("NSG_ASM_DEBUG") ? std::atoi(std::getenv("NSG_ASM_DEBUG")) : 0;
  return P;
}

static int launch_assembly(nsg_ctx *c) {
  const AsmParams P = asm_params(c);
  // The pressure rows of J and Mp depend on the geometry and nu only: they are integrated once and kept while
  // c->p_rows_valid holds (see nsg_ctx).  R_p = 0 is written in every assembly, by the pressure kernel or here.
  const bool run_p = !c->p_rows_valid;
  if (!run_p && c->n_own_p > 0) NSG_CUDA(cudaMemsetAsync(c->R + c->n_own_u, 0, 8 * (size_t)c->n_own_p, c->stream));
  if (c->asm_variant == 5) {
    // fan scheme.  The pressure rows run on a second stream beside the packet pre-pass and the velocity rows
    // (NSG_ASM_CONCURRENT=0: one stream)
    const bool fork = run_p && c->wl_p6.n_chunks > 0 && c->aux_stream && !(std::getenv("NSG_ASM_CONCURRENT") && std::atoi(std::getenv("NSG_ASM_CONCURRENT")) == 0);
    cudaStream_t ps = fork ? c->aux_stream : c->stream;
    if (fork) {
      NSG_CUDA(cudaEventRecord(c->ev_fork, c->stream));
      NSG_CUDA(cudaStreamWaitEvent(c->aux_stream, c->ev_fork, 0));
    }
    auto launch_p = [&]() -> int {
      if (run_p && c->wl_p6.n_chunks > 0) {
        k_assemble_p6<<<(unsigned)c->wl_p6.n_chunks, NPC6, sizeof(double) * (size_t)c->wl_p6.max_stage, ps>>>(
            c->wl_p6, c->n_own_u, c->vals, c->pm_vals, c->R, c->geom8, P);
        NSG_LAUNCH_CHECK(c);
      }
      return NSG_OK;
    };
    if (fork) {
      NSG_TRY(launch_p());
      NSG_CUDA(cudaEventRecord(c->ev_join, c->aux_stream));
    }
    if (c->n_cells > 0) {
      k_cell_packets6<<<(unsigned)((c->n_cells + 127) / 128), 128, 0, c->stream>>>(c->n_cells, c->geom8, c->cell_dofs, c->sol, c->sol_old, P,
                                                                                  c->cellpk);
      NSG_LAUNCH_CHECK(c);
    }
    if (c->wl_u6.n_chunks > 0) {
      static const int minb = std::getenv("NSG_ASM6_MINB") ? std::atoi(std::getenv("NSG_ASM6_MINB")) : 4;
      const unsigned grid = (unsigned)c->wl_u6.n_chunks;
      const size_t smem = sizeof(double) * (size_t)c->wl_u6.max_stage;
      if (minb == 5)
        k_assemble_u6<5><<<grid, NPC6, smem, c->stream>>>(c->wl_u6, c->vals, c->R, c->cellpk, c->geom8, P, c->asm_pf_rec, c->asm_pf_pk);
      else if (minb == 6)
        k_assemble_u6<6><<<grid, NPC6, smem, c->stream>>>(c->wl_u6, c->vals, c->R, c->cellpk, c->geom8, P, c->asm_pf_rec, c->asm_pf_pk);
      else
        k_assemble_u6<4><<<grid, NPC6, smem, c->stream>>>(c->wl_u6, c->vals, c->R, c->cellpk, c->geom8, P, c->asm_pf_rec, c->asm_pf_pk);
      NSG_LAUNCH_CHECK(c);
    }
    if (fork)
      NSG_CUDA(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
    else
      NSG_TRY(launch_p());
  } else if (c->asm_variant == 4) {
    // the pressure rows are integrated on a second stream beside the packet pre-pass and the velocity rows
    // (NSG_ASM_CONCURRENT=0: one stream)
    const bool fork = run_p && c->wl_p5.n_chunks > 0 && c->aux_stream && !(std::getenv("NSG_ASM_CONCURRENT") && std::atoi(std::getenv("NSG_ASM_CONCURRENT")) == 0);
    cudaStream_t ps = fork ? c->aux_stream : c->stream;
    if (fork) {
      NSG_CUDA(cudaEventRecord(c->ev_fork, c->stream));
      NSG_CUDA(cudaStreamWaitEvent(c->aux_stream, c->ev_fork, 0));
    }
    auto launch_p = [&]() -> int {
      if (run_p && c->wl_p5.n_chunks > 0) {
        k_assemble_p5<<<(unsigned)c->wl_p5.n_chunks, NPC5, sizeof(double) * (size_t)c->wl_p5.max_stage, ps>>>(
            c->wl_p5, c->n_own_u, c->vals, c->pm_vals, c->R, c->geom, P);
        NSG_LAUNCH_CHECK(c);
      }
      return NSG_OK;
    };
    if (fork) {
      NSG_TRY(launch_p());
      NSG_CUDA(cudaEventRecord(c->ev_join, c->aux_stream));
    }
    if (c->n_cells > 0) {
      k_cell_packets<<<grid_for(c->n_cells, 128, 1 << 30), 128, 0, c->stream>>>(c->n_cells, c->geom, c->cell_dofs, c->sol, c->sol_old,
                                                                                P, c->cellpk);
      NSG_LAUNCH_CHECK(c);
    }
    if (c->wl_u5.n_chunks > 0) {
      const unsigned grid = (unsigned)c->wl_u5.n_chunks;
      const size_t smem = sizeof(double) * (size_t)c->wl_u5.max_stage;
      const int minb = std::getenv("NSG_ASM3_MINB") ? std::atoi(std::getenv("NSG_ASM3_MINB")) : 4;
      // a CTA pulls the records and packets of the CTA that will follow it on its SM slot towards L2
      const int pf = std::getenv("NSG_ASM_PF") ? std::atoi(std::getenv("NSG_ASM_PF")) : 0;  // measured: no gain (profiles/r01_summary.md)
      if (minb <= 3)
        k_assemble_u5<3><<<grid, NPC5, smem, c->stream>>>(c->wl_u5, c->vals, c->R, c->cellpk, P, pf);
      else if (minb == 4)
        k_assemble_u5<4><<<grid, NPC5, smem, c->stream>>>(c->wl_u5, c->vals, c->R, c->cellpk, P, pf);
      else
        k_assemble_u5<5><<<grid, NPC5, smem, c->stream>>>(c->wl_u5, c->vals, c->R, c->cellpk, P, pf);
      NSG_LAUNCH_CHECK(c);
    }
    if (fork)
      NSG_CUDA(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
    else
      NSG_TRY(launch_p());
  } else {
  if (c->wl_u.n_chunks > 0) {
    k_assemble_u<<<(unsigned)c->wl_u.n_chunks, NPC, sizeof(double) * (size_t)c->wl_u.max_stage, c->stream>>>(
        c->wl_u, c->rowptr, c->vals, c->R, c->geom, c->cell_dofs, c->sol, c->sol_old, P);
    NSG_LAUNCH_CHECK(c);
  }
  if (run_p && c->wl_p.n_chunks > 0) {
    k_assemble_p<<<(unsigned)c->wl_p.n_chunks, NPC, sizeof(double) * (size_t)c->wl_p.max_stage, c->stream>>>(
        c->wl_p, c->n_own_u, c->rowptr, c->vals, c->pm_rowptr, c->pm_vals, c->R, c->geom, P);
    NSG_LAUNCH_CHECK(c);
  }
  }
  if (c->n_bnodes > 0) {
    k_neumann<<<grid_for(c->n_bnodes, 128, 1 << 20), 128, 0, c->stream>>>(c->n_bnodes, c->bnode_dof, c->bnode_ptr, c->bnode_face,
                                                                        c->bnode_pos, c->bface_cell, c->bface_face, c->bface_tag,
                                                                        c->cell_vertices, c->xy, c->R, P);
    NSG_LAUNCH_CHECK(c);
  }
  c->p_rows_valid = true;
  return NSG_OK;
}

// Work lists of the assembly variants 0..3 (slot-based, two pairs per thread): built when one of them is first
// selected, so the default path (variant 4) does not pay their host time and device memory.
static int ensure_slot_worklists(nsg_ctx *c) {
  if (c->wl_u.chunks || c->wl_p.chunks || !c->have_mesh) return NSG_OK;
  std::vector<int32_t> cell_dofs_h((size_t)(15 * c->n_cells));
  NSG_CUDA(cudaMemcpy(cell_dofs_h.data(), c->cell_dofs, sizeof(int32_t) * cell_dofs_h.size(), cudaMemcpyDeviceToHost));
  const int32_t *cell_dofs = cell_dofs_h.data();
  const bool fetch_cols = c->h_col.empty() && c->nnz > 0;  // nsg_set_mesh drops the host copy of the column indices
  if (fetch_cols) {
    c->h_col.resize((size_t)c->nnz), c->h_pm_col.resize((size_t)c->pm_nnz);
    NSG_CUDA(cudaMemcpy(c->h_col.data(), c->col, sizeof(int32_t) * (size_t)c->nnz, cudaMemcpyDeviceToHost));
    NSG_CUDA(cudaMemcpy(c->h_pm_col.data(), c->pm_col, sizeof(int32_t) * (size_t)c->pm_nnz, cudaMemcpyDeviceToHost));
  }
  NSG_TRY(build_worklist(c, 0, cell_dofs, &c->wl_u));
  NSG_TRY(build_worklist(c, 1, cell_dofs, &c->wl_p));
  const size_t smem_u = 8 * (size_t)c->wl_u.max_stage, smem_p = 8 * (size_t)c->wl_p.max_stage;
  if (smem_u > 200 * 1024 || smem_p > 200 * 1024)
    return fail(NSG_ERR_ARG, "a chunk of matrix rows does not fit in shared memory (vertex valence too high)");
  NSG_CUDA(cudaFuncSetAttribute(k_assemble_u, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem_u, 1024)));
  NSG_CUDA(cudaFuncSetAttribute(k_assemble_p, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem_p, 1024)));
  if (fetch_cols) {
    c->h_col.clear(), c->h_col.shrink_to_fit();
    c->h_pm_col.clear(), c->h_pm_col.shrink_to_fit();
  }
  return NSG_OK;
}

// Work lists of assembly variant 4 (round-sorted lanes): built when it is selected or when the fan scheme cannot serve the mesh.
static int ensure_round_worklists(nsg_ctx *c, const int32_t *cell_dofs_host) {
  if (c->wl_u5.chunks || c->wl_p5.chunks || !c->have_mesh) return NSG_OK;
  std::vector<int32_t> cell_dofs_h;
  if (!cell_dofs_host) {
    cell_dofs_h.resize((size_t)(15 * c->n_cells));
    NSG_CUDA(cudaMemcpy(cell_dofs_h.data(), c->cell_dofs, sizeof(int32_t) * cell_dofs_h.size(), cudaMemcpyDeviceToHost));
    cell_dofs_host = cell_dofs_h.data();
  }
  const bool fetch_cols = c->h_col.empty() && c->nnz > 0;
  if (fetch_cols) {
    c->h_col.resize((size_t)c->nnz), c->h_pm_col.resize((size_t)c->pm_nnz);
    NSG_CUDA(cudaMemcpy(c->h_col.data(), c->col, sizeof(int32_t) * (size_t)c->nnz, cudaMemcpyDeviceToHost));
    NSG_CUDA(cudaMemcpy(c->h_pm_col.data(), c->pm_col, sizeof(int32_t) * (size_t)c->pm_nnz, cudaMemcpyDeviceToHost));
  }
  NSG_TRY(build_worklist5(c, 0, cell_dofs_host, &c->wl_u5));
  NSG_TRY(build_worklist5(c, 1, cell_dofs_host, &c->wl_p5));
  const size_t s5u = 8 * (size_t)c->wl_u5.max_stage, s5p = 8 * (size_t)c->wl_p5.max_stage;
  if (s5u > 200 * 1024 || s5p > 200 * 1024)
    return fail(NSG_ERR_ARG, "a chunk of matrix rows does not fit in shared memory (vertex valence too high)");
  NSG_CUDA(cudaFuncSetAttribute(k_assemble_u5<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(s5u, 1024)));
  NSG_CUDA(cudaFuncSetAttribute(k_assemble_u5<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(s5u, 1024)));
  NSG_CUDA(cudaFuncSetAttribute(k_assemble_u5<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(s5u, 1024)));
  NSG_CUDA(cudaFuncSetAttribute(k_assemble_p5, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(s5p, 1024)));
  if (fetch_cols) {
    c->h_col.clear(), c->h_col.shrink_to_fit();
    c->h_pm_col.clear(), c->h_pm_col.shrink_to_fit();
  }
  return NSG_OK;
}

static int ensure_pinned(nsg_ctx *c, int64_t n) {
  if (c->h_pinned_cap >= n) return NSG_OK;
  if (c->h_pinned) cudaFreeHost(c->h_pinned);
  c->h_pinned = nullptr;
  NSG_CUDA(cudaMallocHost((void **)&c->h_pinned, sizeof(double) * (size_t)n));
  c->h_pinned_cap = n;
  return NSG_OK;
}

static bool is_pinned(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}
// host -> device vector of owned length: straight DMA from page-locked caller memory, through the
// context's pinned staging buffer otherwise
static int put_vec(nsg_ctx *c, double *dev, const double *host, int64_t n) {
  const double *src = host;
  if (!is_pinned(host)) {
    NSG_TRY(ensure_pinned(c, n));
    std::memcpy(c->h_pinned, host, sizeof(double) * (size_t)n);
    src = c->h_pinned;
  }
  NSG_CUDA(cudaMemcpyAsync(dev, src, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  c->h2d += 8 * n;
  return NSG_OK;
}
static int get_vec(nsg_ctx *c, const double *dev, double *host, int64_t n) {
  if (is_pinned(host)) {
    NSG_CUDA(cudaMemcpyAsync(host, dev, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    NSG_CUDA(cudaStreamSynchronize(c->stream));
  } else {
    NSG_TRY(ensure_pinned(c, n));
    NSG_CUDA(cudaMemcpyAsync(c->h_pinned, dev, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    NSG_CUDA(cudaStreamSynchronize(c->stream));
    std::memcpy(host, c->h_pinned, sizeof(double) * (size_t)n);
  }
  c->d2h += 8 * n;
  return NSG_OK;
}

}  // namespace nsg

#include "nsg_krylov.cuh"
#include "nsg_precond.cuh"
#include "nsg_gmres_fused.cuh"
#include "nsg_points.cuh"


namespace nsg {
// ---- whole identity-preconditioned GMRES solve as one cooperative kernel (small meshes; nsg_gmres_fused.cuh) ----
static bool gmres_fused_applicable(const nsg_ctx *c, int32_t precond) {
  if (c->gmres_fused == 0 || precond != NSG_PRECOND_IDENTITY || c->n_ranks != 1 || c->orthogonalization != 0) return false;
  if (c->n_own <= 0) return false;
  // one CTA per SM, all co-resident (cooperative launch): the SM count comes from the device (a MIG/MPS slice has fewer
  // than 148), and without cooperative-launch support the multi-kernel solver runs instead
  static int coop = -1;
  if (coop < 0) {
    int v = 0;
    coop = (cudaDeviceGetAttribute(&v, cudaDevAttrCooperativeLaunch, c->device) == cudaSuccess && v) ? 1 : 0;
  }
  if (!coop) return false;
  const int64_t cap = (int64_t)std::min(sm_count(), GF_MAX_GRID) * GF_THREADS * GF_MAX_EPT;
  const int64_t limit = c->gmres_fused == 2 ? cap : c->gmres_fused_max_n;
  return c->n_own <= std::min<int64_t>(limit, cap);
}
static int gmres_fused(nsg_ctx *c, double *x, double rel_tol, int max_steps, int n_tmp, int hist_cap, GmresResult *out) {
  int64_t n = c->n_own;
  const int grid = (int)std::min<int64_t>(std::min(sm_count(), GF_MAX_GRID), (n + GF_THREADS - 1) / GF_THREADS);
  const int64_t T = (int64_t)grid * GF_THREADS;
  const int ept = (int)((n + T - 1) / T);
  if (!c->gf_partials) {  // [2][GF_MAX_GRID] {value, epoch} words + the broadcast word + the epoch counters, zeroed once
    NSG_TRY(dev_alloc(&c->gf_partials, 2 * (2 * GF_MAX_GRID + 1) + 8));
    NSG_CUDA(cudaMemsetAsync(c->gf_partials, 0, sizeof(double) * (2 * (2 * GF_MAX_GRID + 1) + 8), c->stream));
  }
  // tolerance = rel_tol * ||R|| and the scalar state, exactly as gmres_core sets them up
  NSG_TRY(dev_dot(c, n, c->R, c->R, &c->ctl->nrm2, nullptr));
  k_gmres_init<<<1, 1, 0, c->stream>>>(c->ctl, rel_tol, max_steps, n_tmp, hist_cap);
  NSG_LAUNCH_CHECK(c);
  const int64_t *rowptr = c->rowptr;
  const int32_t *col = c->col;
  const double *vals = c->vals, *b = c->R;
  double *basis = c->basis, *hist = c->hist;
  ulonglong2 *slots = reinterpret_cast<ulonglong2 *>(c->gf_partials);
  unsigned long long *epoch_ctr = reinterpret_cast<unsigned long long *>(c->gf_partials + 2 * (2 * GF_MAX_GRID + 1));
  int64_t S = c->stride;
  GmresCtl *ctl = c->ctl;
  void *args[] = {&n, &rowptr, &col, &vals, &x, &b, &basis, &S, &n_tmp, &ctl, &hist, &slots, &epoch_ctr};
  const void *fn = ept <= 1 ? (const void *)k_gmres_solve_fused<1>
                 : ept <= 2 ? (const void *)k_gmres_solve_fused<2>
                 : ept <= 4 ? (const void *)k_gmres_solve_fused<4>
                            : (const void *)k_gmres_solve_fused<8>;
  int per_sm = 0;
  NSG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, GF_THREADS, 0));
  if (per_sm < 1 || grid > per_sm * sm_count()) return fail(NSG_ERR_CUDA, "the fused GMRES kernel cannot be co-resident on this device");
  NSG_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(GF_THREADS), args, 0, c->stream));
  c->launches++;
  NSG_TRY(read_ctl_header(c, c->ctl, c->h_ctl));
  out->its = c->h_ctl->accumulated;
  out->res = c->h_ctl->rho;
  out->ok = (c->h_ctl->state & 0xff) == 1;
  return NSG_OK;
}
}  // namespace nsg

using namespace nsg;

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char *nsg_last_error(void) { return g_err.c_str(); }

void nsg_params_default(nsg_params *p) {
  if (!p) return;
  p->nu = 0.001, p->rho = 1.0, p->p_out = 10.0;  // hpp:703-709
  p->deltat = 0.05;                              // main.cpp:13
  p->forcing[0] = 0.0, p->forcing[1] = -0.0;     // hpp:438: g = 0
  p->neumann_id = 10;                            // cpp:320
  p->use_mass = 1, p->stokes = 0, p->dirichlet_diag = 0;
}

int nsg_create(int device, nsg_ctx **out) {
  if (!out) return fail(NSG_ERR_ARG, "null out pointer");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(NSG_ERR_CUDA, std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(NSG_ERR_ARG, "device ordinal out of range");
  NSG_CUDA(cudaSetDevice(device));
  auto *c = new nsg_ctx;
  c->device = device;
  c->peer.n_ranks = 1;
  if (const char *v = std::getenv("NSG_ASM_VARIANT")) c->asm_variant = (std::atoi(v) == 0 || std::atoi(v) == 4) ? std::atoi(v) : 5;
  nsg_params_default(&c->prm);
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete c;
    return fail(NSG_ERR_CUDA, "cudaStreamCreate failed");
  }
  c->stream = c->own_stream;
  cudaEventCreate(&c->ev0);
  cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking);
  cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming);
  cudaEventCreate(&c->ev1);
  int rc = upload_tables();
  if (rc == NSG_OK) rc = dev_alloc(&c->partials, RED_MAX_BLOCKS);
  if (rc == NSG_OK) rc = dev_alloc(&c->partials_k, (int64_t)CGS_MAXK * RED_MAX_BLOCKS);
  if (rc == NSG_OK) rc = dev_alloc(&c->ticket, 4);
  if (rc == NSG_OK) rc = dev_alloc(&c->scal, 64);
  if (rc == NSG_OK) rc = dev_alloc(&c->ctl, 1);
  if (rc == NSG_OK && cudaMallocHost((void **)&c->h_ctl, sizeof(GmresCtl)) != cudaSuccess) rc = fail(NSG_ERR_CUDA, "cudaMallocHost failed");
  if (rc == NSG_OK) {
    cudaMemset(c->ticket, 0, 16);
    cudaMemset(c->scal, 0, 64 * 8);
    cudaMemset(c->ctl, 0, sizeof(GmresCtl));
  }
  if (rc != NSG_OK) {
    nsg_destroy(c);
    return rc;
  }
  *out = c;
  return NSG_OK;
}

void nsg_destroy(nsg_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto &e : c->graphs) cudaGraphExecDestroy(e.exec);
  c->graphs.clear();
  for (void *m : c->peer_mapped)
    if (m) cudaIpcCloseMemHandle(m);
  dev_free(c->mailbox), dev_free(c->ar_seq), dev_free(c->gf_partials);
  dev_free(c->send_dst), dev_free(c->halo_ctr), dev_free(c->halo_ticket), dev_free(c->halo_err), dev_free(c->bgroups);
  if (c->comm) nccl_api().CommDestroy(c->comm);
  dev_free(c->rowptr), dev_free(c->pm_rowptr), dev_free(c->col), dev_free(c->pm_col), dev_free(c->vals), dev_free(c->pm_vals);
  dev_free(c->spmv_chunk_rows), dev_free(c->diag_pos), dev_free(c->first_idx), dev_free(c->geom), dev_free(c->cellpk), dev_free(c->xy), dev_free(c->cell_vertices), dev_free(c->cell_dofs);
  free_worklist(c->wl_u), free_worklist(c->wl_p), free_worklist(c->wl_u5), free_worklist(c->wl_p5);
  free_worklist(c->wl_u6), free_worklist(c->wl_p6);
  dev_free(c->geom8);
  pt_free(c);
  dev_free(c->bnode_dof), dev_free(c->bnode_ptr), dev_free(c->bnode_face), dev_free(c->bnode_pos);
  dev_free(c->bface_cell), dev_free(c->bface_face), dev_free(c->bface_tag);
  dev_free(c->sol), dev_free(c->sol_old), dev_free(c->delta), dev_free(c->R), dev_free(c->basis), dev_free(c->work);
  dev_free(c->partials), dev_free(c->partials_k), dev_free(c->ticket), dev_free(c->scal), dev_free(c->ctl), dev_free(c->hist);
  dev_free(c->dir_dofs), dev_free(c->dir_vals), dev_free(c->send_idx), dev_free(c->recv_idx), dev_free(c->send_buf), dev_free(c->recv_buf);
  free_blocks(c);
  if (c->h_ctl) cudaFreeHost(c->h_ctl);
  if (c->h_pinned) cudaFreeHost(c->h_pinned);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

int nsg_set_stream(nsg_ctx *c, void *s) {
  if (!c) return fail(NSG_ERR_ARG, "null context");
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  c->stream = s ? (cudaStream_t)s : c->own_stream;
  return NSG_OK;
}

// sizes of a pattern call, common to the two ways a pattern can arrive
static int pattern_sizes(nsg_ctx *c, int64_t n_own_u, int64_t n_own_p, int64_t n_ghost_u, int64_t n_ghost_p) {
  if (n_own_u < 0 || n_own_p < 0 || (n_own_u & 1)) return fail(NSG_ERR_ARG, "n_own_u must be even and sizes non-negative");
  if (c->have_pattern) return fail(NSG_ERR_STATE, "pattern already set (the CSR is fixed for the life of the context)");
  NSG_CUDA(cudaSetDevice(c->device));
  c->n_own_u = n_own_u, c->n_own_p = n_own_p, c->n_own = n_own_u + n_own_p;
  c->n_ghost_u = n_ghost_u, c->n_ghost_p = n_ghost_p;
  c->n_loc = c->n_own + n_ghost_u + n_ghost_p;
  if (c->n_loc >= (int64_t)INT32_MAX) return fail(NSG_ERR_ARG, "local DoF count exceeds 32-bit column indices");
  c->stride = (c->n_loc + 31) / 32 * 32;
  return NSG_OK;
}
// everything after the device CSR (rowptr, col, pm_rowptr, pm_col) and c->h_rowptr / c->h_pm_rowptr exist
static int finish_pattern(nsg_ctx *c, Trace &tr) {
  const int64_t n = c->n_own;
  NSG_TRY(dev_alloc(&c->vals, c->nnz + 16));
  NSG_TRY(dev_alloc(&c->pm_vals, c->pm_nnz));
  NSG_CUDA(cudaMemsetAsync(c->vals, 0, 8 * (size_t)std::max<int64_t>(c->nnz, 1), c->stream));
  NSG_CUDA(cudaMemsetAsync(c->pm_vals, 0, 8 * (size_t)std::max<int64_t>(c->pm_nnz, 1), c->stream));
  NSG_TRY(dev_alloc(&c->diag_pos, n));
  NSG_TRY(dev_alloc(&c->first_idx, 2));
  if (n > 0) {
    k_diag_pos<<<grid_for(n, 256, 1 << 30), 256, 0, c->stream>>>(n, c->rowptr, c->col, c->diag_pos);
    NSG_LAUNCH_CHECK(c);
  }
  std::vector<int32_t> chunks;
  make_spmv_chunks(c->h_rowptr.data(), n, chunks);
  c->spmv_n_chunks = (int64_t)chunks.size() - 1;
  NSG_TRY(upload(c, &c->spmv_chunk_rows, chunks.data(), (int64_t)chunks.size()));
  tr.mark("values, diagonal positions, spmv chunks");
  for (double **v : {&c->sol, &c->sol_old, &c->delta, &c->R}) {
    NSG_TRY(dev_alloc(v, c->stride));
    NSG_CUDA(cudaMemsetAsync(*v, 0, 8 * (size_t)c->stride, c->stream));
  }
  NSG_TRY(dev_alloc(&c->work, 8 * c->stride));
  NSG_CUDA(cudaMemsetAsync(c->work, 0, 8 * 8 * (size_t)c->stride, c->stream));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  tr.mark("vectors + sync");
  c->have_pattern = true;
  return NSG_OK;
}

int nsg_set_pattern(nsg_ctx *c, int64_t n_own_u, int64_t n_own_p, int64_t n_ghost_u, int64_t n_ghost_p,
                    const int64_t *jac_rowptr, const int32_t *jac_col, const int64_t *pm_rowptr, const int32_t *pm_col) {
  if (!c || !jac_rowptr || !jac_col || !pm_rowptr || !pm_col) return fail(NSG_ERR_ARG, "null argument");
  NSG_TRY(pattern_sizes(c, n_own_u, n_own_p, n_ghost_u, n_ghost_p));
  const int64_t n = c->n_own;
  c->nnz = jac_rowptr[n], c->pm_nnz = pm_rowptr[n];
  for (int64_t i = 0; i < n; ++i)
    if (jac_rowptr[i + 1] < jac_rowptr[i] || pm_rowptr[i + 1] < pm_rowptr[i]) return fail(NSG_ERR_ARG, "row pointers not monotone");
  c->h_rowptr.assign(jac_rowptr, jac_rowptr + n + 1);
  Trace tr("nsg_set_pattern");
  c->h_col.assign(jac_col, jac_col + c->nnz);
  c->h_pm_rowptr.assign(pm_rowptr, pm_rowptr + n + 1);
  c->h_pm_col.assign(pm_col, pm_col + c->pm_nnz);
  // +16 elements of slack behind the arrays
  NSG_TRY(dev_alloc(&c->rowptr, n + 1 + 16));
  NSG_CUDA(cudaMemsetAsync(c->rowptr, 0, 8 * (size_t)(n + 17), c->stream));
  NSG_CUDA(cudaMemcpyAsync(c->rowptr, jac_rowptr, 8 * (size_t)(n + 1), cudaMemcpyHostToDevice, c->stream));
  NSG_TRY(dev_alloc(&c->col, c->nnz + 16));
  NSG_CUDA(cudaMemsetAsync(c->col, 0, 4 * (size_t)(c->nnz + 16), c->stream));
  NSG_CUDA(cudaMemcpyAsync(c->col, jac_col, 4 * (size_t)c->nnz, cudaMemcpyHostToDevice, c->stream));
  c->h2d += 8 * (n + 1) + 4 * c->nnz;
  NSG_TRY(upload(c, &c->pm_rowptr, pm_rowptr, n + 1));
  NSG_TRY(upload(c, &c->pm_col, pm_col, c->pm_nnz));
  tr.mark("host copies + uploads queued");
  c->have_paired = rows_come_in_pairs(c, jac_rowptr, jac_col);
  if (c->have_paired && n_ghost_u + n_ghost_p > 0) {  // row groups of SpMV variant 7 that read a ghost column
    const int64_t n_ug = n_own_u / 2, n_groups = n_ug + n_own_p;
    std::vector<uint8_t> flag((size_t)n_groups, 0);
#pragma omp parallel for schedule(static)
    for (int64_t g = 0; g < n_groups; ++g) {
      const int64_t r = g < n_ug ? 2 * g : g + n_ug;
      // columns ascend: ghosts, if any, are at the end of the row
      if (jac_rowptr[r + 1] > jac_rowptr[r] && jac_col[jac_rowptr[r + 1] - 1] >= n) flag[g] = 1;
    }
    std::vector<int32_t> list;
    for (int64_t g = 0; g < n_groups; ++g)
      if (flag[g]) list.push_back((int32_t)g);
    c->n_bgroups = (int64_t)list.size();
    NSG_TRY(upload(c, &c->bgroups, list.data(), c->n_bgroups));
  }
  c->spmv_variant = c->have_paired ? 7 : 4;  // fastest measured (profiles/r01_summary.md); 7 needs the node-pair row structure
  tr.mark("row-pair check");
  return finish_pattern(c, tr);
}

// SURVEY 8f N4: the same two patterns built on the device from the cell -> dof table (nsg_pattern.cuh)
int nsg_set_pattern_from_cells(nsg_ctx *c, int64_t n_own_u, int64_t n_own_p, int64_t n_ghost_u, int64_t n_ghost_p, int64_t n_cells,
                               const int32_t *cell_dofs) {
  if (!c || (n_cells > 0 && !cell_dofs) || n_cells < 0) return fail(NSG_ERR_ARG, "bad argument");
  NSG_TRY(pattern_sizes(c, n_own_u, n_own_p, n_ghost_u, n_ghost_p));
  Trace tr("nsg_set_pattern_from_cells");
  const int64_t n = c->n_own, n_ug = n_own_u / 2, n_groups = n_ug + n_own_p, T = n_cells;
  int32_t *d_cd = nullptr, *gcount = nullptr, *gcells = nullptr, *rowlen = nullptr, *pm_rowlen = nullptr, *err = nullptr;
  int64_t *gptr = nullptr, *tmp = nullptr;
  uint8_t *flag = nullptr;
  auto cleanup = [&]() {
    dev_free(d_cd), dev_free(gcount), dev_free(gcells), dev_free(rowlen), dev_free(pm_rowlen), dev_free(err), dev_free(gptr), dev_free(tmp);
    dev_free(flag);
  };
  auto body = [&]() -> int {
    NSG_TRY(upload(c, &d_cd, cell_dofs, 15 * T));
    NSG_TRY(dev_alloc(&gcount, 2 * n_groups + 2));  // counts, then the fill cursors
    NSG_TRY(dev_alloc(&gptr, n_groups + 1));
    NSG_TRY(dev_alloc(&tmp, 3 * (std::max(n, n_groups) / SCAN_B + 2) + 256));
    NSG_TRY(dev_alloc(&err, 1));
    NSG_CUDA(cudaMemsetAsync(gcount, 0, 4 * (size_t)(2 * n_groups + 2), c->stream));
    NSG_CUDA(cudaMemsetAsync(err, 0, 4, c->stream));
    if (T > 0) {
      k_pat_count<<<grid_for(9 * T, 256, 1 << 30), 256, 0, c->stream>>>(T, d_cd, n_own_u, n, gcount);
      NSG_LAUNCH_CHECK(c);
    }
    NSG_TRY(dev_exclusive_scan<int32_t>(c, n_groups, gcount, gptr, tmp));
    int64_t n_inc = 0;
    NSG_CUDA(cudaMemcpyAsync(&n_inc, gptr + n_groups, 8, cudaMemcpyDeviceToHost, c->stream));
    NSG_CUDA(cudaStreamSynchronize(c->stream));
    NSG_TRY(dev_alloc(&gcells, n_inc));
    if (T > 0) {
      k_pat_fill<<<grid_for(9 * T, 256, 1 << 30), 256, 0, c->stream>>>(T, d_cd, n_own_u, n, gptr, gcount + n_groups + 1, gcells);
      NSG_LAUNCH_CHECK(c);
    }
    tr.mark("group -> cells lists");
    NSG_TRY(dev_alloc(&rowlen, n + 1));
    NSG_TRY(dev_alloc(&pm_rowlen, n + 1));
    if (n_groups > 0) {
      k_pat_rowlen<<<grid_for(n_groups, 128, 1 << 30), 128, 0, c->stream>>>(n_groups, n_ug, gptr, gcells, d_cd, rowlen, pm_rowlen, err);
      NSG_LAUNCH_CHECK(c);
    }
    NSG_TRY(dev_alloc(&c->rowptr, n + 1 + 16));
    NSG_CUDA(cudaMemsetAsync(c->rowptr, 0, 8 * (size_t)(n + 17), c->stream));
    NSG_TRY(dev_alloc(&c->pm_rowptr, n + 1));
    NSG_TRY(dev_exclusive_scan<int32_t>(c, n, rowlen, c->rowptr, tmp));
    NSG_TRY(dev_exclusive_scan<int32_t>(c, n, pm_rowlen, c->pm_rowptr, tmp));
    c->h_rowptr.resize((size_t)n + 1), c->h_pm_rowptr.resize((size_t)n + 1);
    NSG_CUDA(cudaMemcpyAsync(c->h_rowptr.data(), c->rowptr, 8 * (size_t)(n + 1), cudaMemcpyDeviceToHost, c->stream));
    NSG_CUDA(cudaMemcpyAsync(c->h_pm_rowptr.data(), c->pm_rowptr, 8 * (size_t)(n + 1), cudaMemcpyDeviceToHost, c->stream));
    int32_t h_err = 0;
    NSG_CUDA(cudaMemcpyAsync(&h_err, err, 4, cudaMemcpyDeviceToHost, c->stream));
    NSG_CUDA(cudaStreamSynchronize(c->stream));
    c->d2h += 16 * (n + 1);
    if (h_err) return fail(NSG_ERR_ARG, "a patch has more nodes than the device pattern builder holds (104 velocity nodes, 40 pressure vertices: vertex valence <= 34 inside the domain, <= 33 on the boundary)");
    c->nnz = c->h_rowptr[n], c->pm_nnz = c->h_pm_rowptr[n];
    tr.mark("row lengths + scans");
    NSG_TRY(dev_alloc(&c->col, c->nnz + 16));
    NSG_CUDA(cudaMemsetAsync(c->col + c->nnz, 0, 4 * 16, c->stream));
    NSG_TRY(dev_alloc(&c->pm_col, c->pm_nnz));
    if (n_groups > 0) {
      k_pat_cols<<<grid_for(n_groups, 128, 1 << 30), 128, 0, c->stream>>>(n_groups, n_ug, gptr, gcells, d_cd, c->rowptr, c->col, c->pm_rowptr,
                                                                        c->pm_col);
      NSG_LAUNCH_CHECK(c);
    }
    c->have_paired = true;  // by construction: rows 2g and 2g+1 get the same list
    if (n_ghost_u + n_ghost_p > 0 && n_groups > 0) {
      NSG_TRY(dev_alloc(&flag, n_groups));
      k_pat_ghost_flag<<<grid_for(n_groups, 256, 1 << 30), 256, 0, c->stream>>>(n_groups, n_ug, n, c->rowptr, c->col, flag);
      NSG_LAUNCH_CHECK(c);
      std::vector<uint8_t> h_flag((size_t)n_groups);
      NSG_CUDA(cudaMemcpyAsync(h_flag.data(), flag, (size_t)n_groups, cudaMemcpyDeviceToHost, c->stream));
      NSG_CUDA(cudaStreamSynchronize(c->stream));
      std::vector<int32_t> list;
      for (int64_t g = 0; g < n_groups; ++g)
        if (h_flag[g]) list.push_back((int32_t)g);
      c->n_bgroups = (int64_t)list.size();
      NSG_TRY(upload(c, &c->bgroups, list.data(), c->n_bgroups));
    }
    c->spmv_variant = 7;
    c->pattern_on_device = true;  // no host copy of the column indices: the fan lists look their offsets up on the device
    tr.mark("columns");
    return NSG_OK;
  };
  const int rc = body();
  cudaStreamSynchronize(c->stream);
  cleanup();
  if (rc != NSG_OK) return rc;
  return finish_pattern(c, tr);
}

int nsg_get_pattern_sizes(nsg_ctx *c, int64_t *nnz_jac, int64_t *nnz_pm) {
  if (!c || !c->have_pattern) return fail(NSG_ERR_STATE, "no pattern");
  if (nnz_jac) *nnz_jac = c->nnz;
  if (nnz_pm) *nnz_pm = c->pm_nnz;
  return NSG_OK;
}
int nsg_get_pattern(nsg_ctx *c, int64_t *jac_rowptr, int32_t *jac_col, int64_t *pm_rowptr, int32_t *pm_col) {
  if (!c || !c->have_pattern) return fail(NSG_ERR_STATE, "no pattern");
  NSG_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n_own;
  if (jac_rowptr) NSG_CUDA(cudaMemcpy(jac_rowptr, c->rowptr, 8 * (size_t)(n + 1), cudaMemcpyDeviceToHost));
  if (jac_col && c->nnz > 0) NSG_CUDA(cudaMemcpy(jac_col, c->col, 4 * (size_t)c->nnz, cudaMemcpyDeviceToHost));
  if (pm_rowptr) NSG_CUDA(cudaMemcpy(pm_rowptr, c->pm_rowptr, 8 * (size_t)(n + 1), cudaMemcpyDeviceToHost));
  if (pm_col && c->pm_nnz > 0) NSG_CUDA(cudaMemcpy(pm_col, c->pm_col, 4 * (size_t)c->pm_nnz, cudaMemcpyDeviceToHost));
  return NSG_OK;
}

int nsg_set_mesh(nsg_ctx *c, int64_t n_cells, int64_t n_vertices, const double *xy, const int32_t *cell_vertices,
                 const int32_t *cell_dofs, int64_t n_bfaces, const int32_t *bface_cell, const int32_t *bface_face,
                 const int32_t *bface_tag) {
  if (!c || !xy || !cell_vertices || !cell_dofs) return fail(NSG_ERR_ARG, "null argument");
  if (!c->have_pattern) return fail(NSG_ERR_STATE, "nsg_set_pattern must be called before nsg_set_mesh");
  if (c->have_mesh) return fail(NSG_ERR_STATE, "mesh already set");
  if (n_bfaces > 0 && (!bface_cell || !bface_face || !bface_tag)) return fail(NSG_ERR_ARG, "null boundary-face arrays");
  NSG_CUDA(cudaSetDevice(c->device));
  Trace tr("nsg_set_mesh");
  for (int64_t i = 0; i < 15 * n_cells; ++i)
    if (cell_dofs[i] < 0 || cell_dofs[i] >= c->n_loc) return fail(NSG_ERR_ARG, "cell_dofs entry out of range");
  for (int64_t i = 0; i < 3 * n_cells; ++i)
    if (cell_vertices[i] < 0 || cell_vertices[i] >= n_vertices) return fail(NSG_ERR_ARG, "cell_vertices entry out of range");
  c->n_cells = n_cells, c->n_vertices = n_vertices, c->n_bfaces = n_bfaces;
  NSG_TRY(upload(c, &c->xy, xy, 2 * n_vertices));
  NSG_TRY(upload(c, &c->cell_vertices, cell_vertices, 3 * n_cells));
  NSG_TRY(upload(c, &c->cell_dofs, cell_dofs, 15 * n_cells));
  NSG_TRY(upload(c, &c->bface_cell, bface_cell, n_bfaces));
  NSG_TRY(upload(c, &c->bface_face, bface_face, n_bfaces));
  NSG_TRY(upload(c, &c->bface_tag, bface_tag, n_bfaces));
  NSG_TRY(dev_alloc(&c->geom, 5 * n_cells));
  if (n_cells > 0) {
    k_cell_geometry<<<grid_for(n_cells, 256, 1 << 30), 256, 0, c->stream>>>(n_cells, c->xy, c->cell_vertices, c->geom);
    NSG_LAUNCH_CHECK(c);
  }
  NSG_TRY(dev_alloc(&c->geom8, 8 * n_cells));
  if (n_cells > 0) {
    k_cell_geometry8<<<grid_for(n_cells, 256, 1 << 30), 256, 0, c->stream>>>(n_cells, c->xy, c->cell_vertices, c->geom8);
    NSG_LAUNCH_CHECK(c);
  }
  NSG_TRY(dev_alloc(&c->cellpk, PK * n_cells + 2));
  // default: the fan scheme (variant 5); its lists exist only for oriented manifold triangulations.  The work lists of
  // the other variants are built on demand (nsg_set_tuning key 1) or when the fan scheme cannot serve the mesh.
  {
    bool ok_u = false, ok_p = false;
    tr.mark("checks + uploads + geometry");
    NSG_TRY(build_fanlist(c, 0, cell_dofs, &c->wl_u6, &ok_u));
    tr.mark("fan list (velocity rows)");
    if (ok_u) NSG_TRY(build_fanlist(c, 1, cell_dofs, &c->wl_p6, &ok_p));
    tr.mark("fan list (pressure rows)");
    const size_t s6u = 8 * (size_t)c->wl_u6.max_stage, s6p = 8 * (size_t)c->wl_p6.max_stage;
    c->fan_ok = ok_u && ok_p && s6u <= 200 * 1024 && s6p <= 200 * 1024;
    if (c->fan_ok) {
      NSG_CUDA(cudaFuncSetAttribute(k_assemble_u6<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(s6u, 1024)));
      NSG_CUDA(cudaFuncSetAttribute(k_assemble_u6<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(s6u, 1024)));
    } else {
      free_worklist(c->wl_u6), free_worklist(c->wl_p6);
      if (c->asm_variant == 5) {
        // the fallback: variant 4 up to ASM_MAX_VALENCE_4 cells per row owner, variant 0 up to ASM_MAX_VALENCE_0
        const int v = max_owner_cells(c, cell_dofs);
        if (v > ASM_MAX_VALENCE_0)
          return fail(NSG_ERR_ARG, "a vertex has " + std::to_string(v) + " incident cells: the assembly serves at most " +
                                       std::to_string(ASM_MAX_VALENCE_0));
        c->asm_variant = v <= ASM_MAX_VALENCE_4 ? 4 : 0;
      }
    }
  }
  // Neumann: owned boundary P2 nodes -> (face, position on the face)
  {
    struct Ent {
      int32_t dof, face, pos;
    };
    std::vector<Ent> ents;
    for (int64_t i = 0; i < n_bfaces; ++i) {
      const int64_t cell = bface_cell[i];
      const int f = bface_face[i];
      if (cell < 0 || cell >= n_cells || f < 0 || f > 2) return fail(NSG_ERR_ARG, "boundary face out of range");
      const int ks[3] = {f, (f + 1) % 3, 3 + f};
      for (int pos = 0; pos < 3; ++pos) {
        const int32_t d = cell_dofs[15 * cell + uidx(ks[pos])];
        if (d < c->n_own_u) ents.push_back({d, (int32_t)i, pos});
      }
    }
    std::stable_sort(ents.begin(), ents.end(), [](const Ent &a, const Ent &b) { return a.dof < b.dof; });
    std::vector<int32_t> ndof, nptr{0}, nface, npos;
    for (size_t i = 0; i < ents.size(); ++i) {
      if (i == 0 || ents[i].dof != ents[i - 1].dof) {
        if (i) nptr.push_back((int32_t)i);
        ndof.push_back(ents[i].dof);
      }
      nface.push_back(ents[i].face);
      npos.push_back(ents[i].pos);
    }
    nptr.push_back((int32_t)ents.size());
    c->n_bnodes = (int64_t)ndof.size();
    NSG_TRY(upload(c, &c->bnode_dof, ndof.data(), (int64_t)ndof.size()));
    NSG_TRY(upload(c, &c->bnode_ptr, nptr.data(), (int64_t)nptr.size()));
    NSG_TRY(upload(c, &c->bnode_face, nface.data(), (int64_t)nface.size()));
    NSG_TRY(upload(c, &c->bnode_pos, npos.data(), (int64_t)npos.size()));
    NSG_CUDA(cudaStreamSynchronize(c->stream));
  }
  c->have_mesh = true;
  if (c->asm_variant == 4) {
    NSG_TRY(ensure_round_worklists(c, cell_dofs));
  } else if (c->asm_variant < 4) {
    NSG_TRY(ensure_slot_worklists(c));
  }
  c->h_col.clear(), c->h_col.shrink_to_fit();
  c->h_pm_col.clear(), c->h_pm_col.shrink_to_fit();
  return NSG_OK;
}

int nsg_set_halo(nsg_ctx *c, int32_t n_neighbors, const int32_t *neighbors, const int64_t *send_ptr, const int32_t *send_idx,
                 const int64_t *recv_ptr, const int32_t *recv_idx) {
  if (!c || n_neighbors < 0) return fail(NSG_ERR_ARG, "bad argument");
  if (!c->have_pattern) return fail(NSG_ERR_STATE, "nsg_set_pattern first");
  c->n_neighbors = n_neighbors;
  if (n_neighbors == 0) return NSG_OK;
  if (!neighbors || !send_ptr || !send_idx || !recv_ptr || !recv_idx) return fail(NSG_ERR_ARG, "null argument");
  c->neighbors.assign(neighbors, neighbors + n_neighbors);
  c->send_ptr.assign(send_ptr, send_ptr + n_neighbors + 1);
  c->recv_ptr.assign(recv_ptr, recv_ptr + n_neighbors + 1);
  c->n_send = send_ptr[n_neighbors], c->n_recv = recv_ptr[n_neighbors];
  for (int64_t i = 0; i < c->n_send; ++i)
    if (send_idx[i] < 0 || send_idx[i] >= c->n_own) return fail(NSG_ERR_ARG, "send index is not an owned DoF");
  for (int64_t i = 0; i < c->n_recv; ++i)
    if (recv_idx[i] < c->n_own || recv_idx[i] >= c->n_loc) return fail(NSG_ERR_ARG, "recv index is not a ghost DoF");
  NSG_TRY(upload(c, &c->send_idx, send_idx, c->n_send));
  NSG_TRY(upload(c, &c->recv_idx, recv_idx, c->n_recv));
  NSG_TRY(dev_alloc(&c->send_buf, c->n_send));
  NSG_TRY(dev_alloc(&c->recv_buf, c->n_recv));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  return NSG_OK;
}

int nsg_comm_unique_id(void *out128) {
  if (!out128) return fail(NSG_ERR_ARG, "null argument");
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  if (!nccl_api().handle) return fail(NSG_ERR_NCCL, nccl_api().error);
  ncclUniqueId id;
  NSG_NCCL(nccl_api().GetUniqueId(&id));
  std::memcpy(out128, &id, sizeof id);
  return NSG_OK;
}

int nsg_comm_init(nsg_ctx *c, int rank, int n_ranks, const void *unique_id128) {
  if (!c || !unique_id128 || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(NSG_ERR_ARG, "bad argument");
  NSG_CUDA(cudaSetDevice(c->device));
  c->rank = rank, c->n_ranks = n_ranks;
  if (n_ranks == 1) return NSG_OK;
  if (!nccl_api().handle) return fail(NSG_ERR_NCCL, nccl_api().error);
  ncclUniqueId id;
  std::memcpy(&id, unique_id128, sizeof id);
  NSG_NCCL(nccl_api().CommInitRank(&c->comm, n_ranks, id, rank));
  return NSG_OK;
}

int nsg_comm_ipc_handle(nsg_ctx *c, void *out64) {
  if (!c || !out64) return fail(NSG_ERR_ARG, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  NSG_CUDA(cudaSetDevice(c->device));
  if (c->n_ranks > PEER_MAX_RANKS) return fail(NSG_ERR_ARG, "more ranks than mailbox slots");
  // mailbox = [ all-reduce words | halo table | halo inbox (two parities per ghost) ]; (re)made and zeroed on every call, so
  // that no stamp of an earlier session can match (the sequence counters restart at 0 in nsg_comm_set_peers)
  const int64_t bytes = PEER_INBOX_OFFSET + 2 * 16 * std::max<int64_t>(c->n_recv, 1);
  if (c->mailbox && c->mailbox_bytes < bytes) dev_free(c->mailbox);
  if (!c->mailbox) {
    NSG_TRY(dev_alloc(&c->mailbox, bytes));
    c->mailbox_bytes = bytes;
  }
  NSG_CUDA(cudaMemset(c->mailbox, 0, (size_t)c->mailbox_bytes));
  PeerHaloTable tab;
  for (int q = 0; q < PEER_MAX_RANKS; ++q) tab.recv_off[q] = -1, tab.recv_cnt[q] = 0;
  for (int k = 0; k < c->n_neighbors; ++k) {
    const int q = c->neighbors[k];
    if (q < 0 || q >= PEER_MAX_RANKS) return fail(NSG_ERR_ARG, "neighbour rank out of range");
    tab.recv_off[q] = c->recv_ptr[k], tab.recv_cnt[q] = c->recv_ptr[k + 1] - c->recv_ptr[k];
  }
  NSG_CUDA(cudaMemcpy(c->mailbox + PEER_AR_WORDS * 16, &tab, sizeof tab, cudaMemcpyHostToDevice));
  cudaIpcMemHandle_t h;
  NSG_CUDA(cudaIpcGetMemHandle(&h, c->mailbox));
  std::memcpy(out64, &h, sizeof h);
  return NSG_OK;
}

int nsg_comm_set_peers(nsg_ctx *c, const void *handles) {
  if (!c || !handles) return fail(NSG_ERR_ARG, "null argument");
  if (c->n_ranks <= 1) return NSG_OK;
  if (c->n_ranks > PEER_MAX_RANKS) return fail(NSG_ERR_ARG, "more ranks than mailbox slots");
  if (!c->mailbox) return fail(NSG_ERR_STATE, "nsg_comm_ipc_handle must be called first");
  NSG_CUDA(cudaSetDevice(c->device));
  PeerComm pc{};
  pc.rank = c->rank;
  char *base[PEER_MAX_RANKS] = {};
  for (int p = 0; p < c->n_ranks; ++p) {
    if (p == c->rank) {
      base[p] = c->mailbox;
    } else {
      cudaIpcMemHandle_t h;
      std::memcpy(&h, (const char *)handles + 64 * (size_t)p, sizeof h);
      void *ptr = nullptr;
      NSG_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
      c->peer_mapped[p] = ptr;
      base[p] = (char *)ptr;
    }
    pc.ar[p] = reinterpret_cast<PeerWord *>(base[p]);
  }
  if (!c->ar_seq) NSG_TRY(dev_alloc(&c->ar_seq, 1));
  NSG_CUDA(cudaMemset(c->ar_seq, 0, sizeof(unsigned long long)));
  pc.seq_ctr = c->ar_seq;
  // halo over peer stores: where in each neighbour's inbox do my values go? (the neighbour wrote its table before it
  // exported its handle, i.e. before the host gathered the handles)
  c->halo_peer = false;
  if (c->n_neighbors > 0) {
    std::vector<PeerWord *> dst((size_t)std::max<int64_t>(c->n_send, 1), nullptr);
    for (int k = 0; k < c->n_neighbors; ++k) {
      const int q = c->neighbors[k];
      PeerHaloTable tab;
      NSG_CUDA(cudaMemcpy(&tab, base[q] + PEER_AR_WORDS * 16, sizeof tab, cudaMemcpyDeviceToHost));
      const int64_t ns = c->send_ptr[k + 1] - c->send_ptr[k];
      if (tab.recv_off[c->rank] < 0 || tab.recv_cnt[c->rank] != ns)
        return fail(NSG_ERR_ARG, "halo plans of two neighbouring ranks do not match");
      PeerWord *inbox = reinterpret_cast<PeerWord *>(base[q] + PEER_INBOX_OFFSET);
      for (int64_t j = 0; j < ns; ++j) dst[(size_t)(c->send_ptr[k] + j)] = inbox + 2 * (tab.recv_off[c->rank] + j);
    }
    dev_free(c->send_dst);
    NSG_TRY(upload(c, &c->send_dst, dst.data(), (int64_t)dst.size()));
    if (!c->halo_ctr) NSG_TRY(dev_alloc(&c->halo_ctr, 2));
    if (!c->halo_ticket) NSG_TRY(dev_alloc(&c->halo_ticket, 2));
    if (!c->halo_err) NSG_TRY(dev_alloc(&c->halo_err, 1));
    NSG_CUDA(cudaMemsetAsync(c->halo_ctr, 0, 16, c->stream));
    NSG_CUDA(cudaMemsetAsync(c->halo_ticket, 0, 8, c->stream));
    NSG_CUDA(cudaMemsetAsync(c->halo_err, 0, 4, c->stream));
    NSG_CUDA(cudaStreamSynchronize(c->stream));
    c->halo_peer = !(std::getenv("NSG_NO_PEER_HALO") && std::atoi(std::getenv("NSG_NO_PEER_HALO")) != 0);
  }
  pc.n_ranks = c->n_ranks;  // switches the reductions to the fused all-reduce
  c->peer = pc;
  for (auto &e : c->graphs) cudaGraphExecDestroy(e.exec);
  c->graphs.clear();
  return NSG_OK;
}

int nsg_comm_release_peers(nsg_ctx *c) {
  if (!c) return fail(NSG_ERR_ARG, "null context");
  NSG_CUDA(cudaSetDevice(c->device));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  c->peer.n_ranks = 1;  // reductions and the halo exchange go back to NCCL
  c->halo_peer = false;
  for (auto &e : c->graphs) cudaGraphExecDestroy(e.exec);
  c->graphs.clear();
  for (void *&m : c->peer_mapped)
    if (m) {
      cudaIpcCloseMemHandle(m);
      m = nullptr;
    }
  return NSG_OK;
}

int nsg_set_params(nsg_ctx *c, const nsg_params *p) {
  if (!c || !p) return fail(NSG_ERR_ARG, "null argument");
  if (!(p->nu > 0) || (p->use_mass && !(p->deltat > 0))) return fail(NSG_ERR_ARG, "nu and deltat must be positive");
  if (p->dirichlet_diag < 0 || p->dirichlet_diag > 1) return fail(NSG_ERR_ARG, "dirichlet_diag must be 0 (Trilinos rule) or 1 (keep a non-zero diagonal)");
  if (p->nu != c->prm.nu) c->p_rows_valid = false;  // the only parameter the pressure-row kernels read (Mp = table/nu)
  c->prm = *p;
  return NSG_OK;
}

int nsg_assemble(nsg_ctx *c) {
  if (!c) return fail(NSG_ERR_ARG, "null context");
  if (!c->have_mesh) return fail(NSG_ERR_STATE, "nsg_set_pattern and nsg_set_mesh must precede nsg_assemble");
  NSG_CUDA(cudaSetDevice(c->device));
  NSG_CUDA(cudaEventRecord(c->ev0, c->stream));
  NSG_TRY(launch_assembly(c));
  NSG_CUDA(cudaEventRecord(c->ev1, c->stream));
  NSG_CUDA(cudaEventSynchronize(c->ev1));
  float ms = 0;
  cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  c->phase_ms[0] = ms;
  c->blocks_stale = true;
  return NSG_OK;
}

int nsg_apply_dirichlet(nsg_ctx *c, int64_t n, const int32_t *dofs, const double *values, int32_t into_solution) {
  if (!c || n < 0 || (n > 0 && (!dofs || !values))) return fail(NSG_ERR_ARG, "bad argument");
  if (!c->have_mesh) return fail(NSG_ERR_STATE, "nsg_set_mesh first");
  NSG_CUDA(cudaSetDevice(c->device));
  if (n == 0) return NSG_OK;
  for (int64_t i = 0; i < n; ++i)
    if (dofs[i] < 0 || dofs[i] >= c->n_own) return fail(NSG_ERR_ARG, "Dirichlet dof is not a locally owned row");
  if (c->dir_cap < n) {
    dev_free(c->dir_dofs), dev_free(c->dir_vals);
    c->h_dir_dofs.clear(), c->h_dir_vals.clear();
    NSG_TRY(dev_alloc(&c->dir_dofs, n));
    NSG_TRY(dev_alloc(&c->dir_vals, n));
    c->dir_cap = n;
  }
  NSG_CUDA(cudaEventRecord(c->ev0, c->stream));
  // the list is the same in every Newton iteration unless the inlet changes (frozen / constant inlet, SURVEY F3): the copy on the
  // device is reused when the caller passes the same dofs and values again (two small pageable copies cost more than the kernels)
  const bool same_dofs = (int64_t)c->h_dir_dofs.size() == n && std::memcmp(c->h_dir_dofs.data(), dofs, 4 * (size_t)n) == 0;
  const bool same_vals = same_dofs && (int64_t)c->h_dir_vals.size() == n && std::memcmp(c->h_dir_vals.data(), values, 8 * (size_t)n) == 0;
  if (!same_dofs) {
    c->h_dir_dofs.assign(dofs, dofs + n);
    NSG_CUDA(cudaMemcpyAsync(c->dir_dofs, c->h_dir_dofs.data(), 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    c->h2d += 4 * n;
  }
  if (!same_vals) {
    c->h_dir_vals.assign(values, values + n);
    NSG_CUDA(cudaMemcpyAsync(c->dir_vals, c->h_dir_vals.data(), 8 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    c->h2d += 8 * n;
  }
  // d_b = |first non-zero diagonal entry of block (b,b) in the local range|, only for blocks that
  // have constrained rows (the per-block apply_boundary_values returns early otherwise)
  bool has_blk[2] = {false, false};
  for (int64_t i = 0; i < n && !(has_blk[0] && has_blk[1]); ++i) has_blk[dofs[i] < c->n_own_u ? 0 : 1] = true;
  if (has_blk[1]) c->p_rows_valid = false;  // a constrained pressure row: the next assembly integrates the pressure rows again
  NSG_CUDA(cudaMemsetAsync(c->first_idx, 0xff, 16, c->stream));
  for (int b = 0; b < 2; ++b) {
    if (!has_blk[b]) continue;
    const int64_t r0 = b == 0 ? 0 : c->n_own_u, r1 = b == 0 ? c->n_own_u : c->n_own;
    if (r1 > r0) {
      // the answer is almost always among the first rows: a 16-block launch looks at the first 4 096 rows, the launch over the rest
      // returns at once when that found one (every block first compares its base row with the index found so far)
      const int64_t rh = std::min<int64_t>(r0 + 4096, r1);
      k_first_nonzero_diag_index<<<16, 256, 0, c->stream>>>(r0, rh, c->diag_pos, c->vals, c->first_idx + b);
      NSG_LAUNCH_CHECK(c);
      if (r1 > rh) {
        k_first_nonzero_diag_index<<<grid_for(r1 - rh, 256, sm_count() * 8), 256, 0, c->stream>>>(rh, r1, c->diag_pos, c->vals, c->first_idx + b);
        NSG_LAUNCH_CHECK(c);
      }
    }
    k_first_nonzero_diag_value<<<1, 1, 0, c->stream>>>(c->diag_pos, c->vals, c->first_idx + b, c->scal + 8 + b);
    NSG_LAUNCH_CHECK(c);
  }
  // Stokes path (cpp:529): the reference writes the values into the GHOSTED `solution`, which the
  // solve never reads (it iterates on solution_owned) and overwrites afterwards -> no vector write here.
  double *x = into_solution ? nullptr : c->delta;
  k_apply_dirichlet<<<(unsigned)((n * 32 + 127) / 128), 128, 0, c->stream>>>(n, c->dir_dofs, c->dir_vals, c->n_own_u, c->rowptr,
                                                                             c->diag_pos, c->vals, x, c->R, c->scal + 8, c->prm.dirichlet_diag);
  NSG_LAUNCH_CHECK(c);
  NSG_CUDA(cudaEventRecord(c->ev1, c->stream));
  NSG_CUDA(cudaEventSynchronize(c->ev1));  // dofs/values are caller-owned: the copies must have completed
  float ms = 0;
  cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  c->phase_ms[1] = ms;
  c->blocks_stale = true;
  return NSG_OK;
}

int nsg_residual_norm(nsg_ctx *c, double *out) {
  if (!c || !out) return fail(NSG_ERR_ARG, "null argument");
  if (!c->have_pattern) return fail(NSG_ERR_STATE, "nsg_set_pattern first");
  NSG_CUDA(cudaSetDevice(c->device));
  NSG_TRY(dev_dot(c, c->n_own, c->R, c->R, c->scal, nullptr));
  double v = 0;
  NSG_CUDA(cudaMemcpyAsync(&v, c->scal, 8, cudaMemcpyDeviceToHost, c->stream));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  c->d2h += 8;
  *out = std::sqrt(v);
  return NSG_OK;
}

int nsg_solve(nsg_ctx *c, int32_t precond, double rel_tol, int32_t max_it, int32_t n_tmp, int32_t target, int32_t *its_out,
              double *res_out) {
  if (!c) return fail(NSG_ERR_ARG, "null context");
  if (!c->have_mesh) return fail(NSG_ERR_STATE, "nsg_set_mesh first");
  if (n_tmp < 3 || n_tmp > GM_MAX_TMP) return fail(NSG_ERR_ARG, "n_tmp_vectors must be in [3,64]");
  if (precond < 0 || precond > 2 || max_it < 0) return fail(NSG_ERR_ARG, "bad precond / max_it");
  NSG_CUDA(cudaSetDevice(c->device));
  const int64_t S = c->stride;
  if (c->basis_n_tmp < n_tmp) {
    dev_free(c->basis);
    NSG_TRY(dev_alloc(&c->basis, (int64_t)n_tmp * S));
    c->basis_n_tmp = n_tmp;
  }
  const int64_t hist_cap = std::min<int64_t>(max_it, 1 << 22);
  if (c->hist_cap < hist_cap) {
    dev_free(c->hist);
    NSG_TRY(dev_alloc(&c->hist, hist_cap));
    c->hist_cap = hist_cap;
  }
  NSG_CUDA(cudaEventRecord(c->ev0, c->stream));
  if (precond != NSG_PRECOND_IDENTITY) NSG_TRY(precond_initialize(c));
  double *x = target ? c->sol : c->delta;
  Op A = [c](double *d, double *s, const int32_t *state) { return dev_spmv(c, s, d, state); };
  Op P = [c, precond](double *d, double *s, const int32_t *) { return precond_vmult(c, precond, d, s); };
  GmresResult r;
  c->inner_its = 0;
  const bool fused = gmres_fused_applicable(c, precond);
  c->last_solve[0] = fused ? 1 : 0, c->last_solve[1] = 0, c->last_solve[2] = fused ? -1 : c->spmv_variant, c->last_solve[3] = c->orthogonalization;
  if (fused)
    NSG_TRY(gmres_fused(c, x, rel_tol, max_it, n_tmp, (int)hist_cap, &r));
  else
    NSG_TRY(gmres_core(c, Range{0, c->n_own}, A, precond == NSG_PRECOND_IDENTITY ? nullptr : &P, x, c->R, c->R, rel_tol, max_it, n_tmp,
                       c->basis, c->ctl, c->h_ctl, c->hist, (int)hist_cap, precond == NSG_PRECOND_IDENTITY, &r));
  if (its_out) *its_out = r.its;
  if (res_out) *res_out = r.res;
  c->h_hist.resize(std::min<int64_t>(r.its, c->hist_cap));
  if (!c->h_hist.empty()) {
    NSG_CUDA(cudaMemcpyAsync(c->h_hist.data(), c->hist, 8 * c->h_hist.size(), cudaMemcpyDeviceToHost, c->stream));
    c->d2h += 8 * (int64_t)c->h_hist.size();
  }
  // solution = solution_owned (cpp:587 / 556): ghost import
  NSG_TRY(halo_exchange(c, c->sol));
  NSG_CUDA(cudaEventRecord(c->ev1, c->stream));
  NSG_CUDA(cudaEventSynchronize(c->ev1));
  float ms = 0;
  cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  c->phase_ms[2] = ms;
  if (!r.ok) {
    char buf[160];
    snprintf(buf, sizeof buf, "GMRES did not converge: %d steps, last residual %.6e", r.its, r.res);
    return fail(NSG_ERR_NO_CONVERGENCE, buf);
  }
  return NSG_OK;
}

int nsg_last_solve_info(nsg_ctx *c, int32_t *out4) {
  if (!c || !out4) return fail(NSG_ERR_ARG, "null argument");
  for (int i = 0; i < 4; ++i) out4[i] = c->last_solve[i];
  return NSG_OK;
}

int64_t nsg_last_inner_iterations(nsg_ctx *c) { return c ? c->inner_its : 0; }

int64_t nsg_gmres_history(nsg_ctx *c, double *out, int64_t cap) {
  if (!c) return 0;
  const int64_t n = std::min<int64_t>(cap, (int64_t)c->h_hist.size());
  if (out) std::copy(c->h_hist.begin(), c->h_hist.begin() + n, out);
  return (int64_t)c->h_hist.size();
}

int nsg_update_solution(nsg_ctx *c) {
  if (!c || !c->have_pattern) return fail(NSG_ERR_STATE, "context not set up");
  NSG_CUDA(cudaSetDevice(c->device));
  k_sadd<<<grid_for(c->n_own, 256), 256, 0, c->stream>>>(c->n_own, c->sol, 1.0, 1.0, c->delta);
  NSG_LAUNCH_CHECK(c);
  return halo_exchange(c, c->sol);
}

int nsg_push_time_level(nsg_ctx *c) {
  if (!c || !c->have_pattern) return fail(NSG_ERR_STATE, "context not set up");
  NSG_CUDA(cudaSetDevice(c->device));
  NSG_CUDA(cudaMemcpyAsync(c->sol_old, c->sol, 8 * (size_t)c->n_loc, cudaMemcpyDeviceToDevice, c->stream));
  return NSG_OK;
}

static int set_owned(nsg_ctx *c, double *dev, const double *host, bool ghosts) {
  if (!c || !host) return fail(NSG_ERR_ARG, "null argument");
  if (!c->have_pattern) return fail(NSG_ERR_STATE, "nsg_set_pattern first");
  NSG_CUDA(cudaSetDevice(c->device));
  NSG_TRY(put_vec(c, dev, host, c->n_own));
  if (ghosts) {
    NSG_TRY(halo_exchange(c, dev));
    NSG_CUDA(cudaStreamSynchronize(c->stream));
  }
  return NSG_OK;
}
static int get_owned(nsg_ctx *c, const double *dev, double *host, int64_t n) {
  if (!c || !host) return fail(NSG_ERR_ARG, "null argument");
  if (!c->have_pattern) return fail(NSG_ERR_STATE, "nsg_set_pattern first");
  NSG_CUDA(cudaSetDevice(c->device));
  return get_vec(c, dev, host, n);
}
int nsg_set_solution(nsg_ctx *c, const double *h) { return set_owned(c, c ? c->sol : nullptr, h, true); }
int nsg_set_solution_old(nsg_ctx *c, const double *h) { return set_owned(c, c ? c->sol_old : nullptr, h, true); }
int nsg_set_delta(nsg_ctx *c, const double *h) { return set_owned(c, c ? c->delta : nullptr, h, false); }
int nsg_get_solution(nsg_ctx *c, double *h) { return get_owned(c, c ? c->sol : nullptr, h, c ? c->n_own : 0); }
int nsg_get_solution_ghosted(nsg_ctx *c, double *h) { return get_owned(c, c ? c->sol : nullptr, h, c ? c->n_loc : 0); }
int nsg_get_delta(nsg_ctx *c, double *h) { return get_owned(c, c ? c->delta : nullptr, h, c ? c->n_own : 0); }
int nsg_get_residual(nsg_ctx *c, double *h) { return get_owned(c, c ? c->R : nullptr, h, c ? c->n_own : 0); }
int nsg_get_matrix_values(nsg_ctx *c, double *h) { return get_owned(c, c ? c->vals : nullptr, h, c ? c->nnz : 0); }
int nsg_get_pm_values(nsg_ctx *c, double *h) { return get_owned(c, c ? c->pm_vals : nullptr, h, c ? c->pm_nnz : 0); }
int nsg_set_solution_ghosted(nsg_ctx *c, const double *h) {
  if (!c || !h) return fail(NSG_ERR_ARG, "null argument");
  if (!c->have_pattern) return fail(NSG_ERR_STATE, "nsg_set_pattern first");
  NSG_CUDA(cudaSetDevice(c->device));
  return put_vec(c, c->sol, h, c->n_loc);
}

int nsg_spmv(nsg_ctx *c, const double *x, double *y) {
  if (!c || !x || !y) return fail(NSG_ERR_ARG, "null argument");
  if (!c->have_pattern) return fail(NSG_ERR_STATE, "nsg_set_pattern first");
  NSG_CUDA(cudaSetDevice(c->device));
  double *dx = c->work, *dy = c->work + c->stride;
  NSG_TRY(put_vec(c, dx, x, c->n_own));
  NSG_TRY(dev_spmv(c, dx, dy, nullptr));
  return get_vec(c, dy, y, c->n_own);
}

int nsg_precond_apply(nsg_ctx *c, int32_t precond, const double *x, double *y) {
  if (!c || !x || !y) return fail(NSG_ERR_ARG, "null argument");
  if (!c->have_mesh) return fail(NSG_ERR_STATE, "nsg_set_mesh first");
  NSG_CUDA(cudaSetDevice(c->device));
  double *dx = c->work, *dy = c->work + c->stride;
  NSG_TRY(put_vec(c, dx, x, c->n_own));
  NSG_CUDA(cudaMemsetAsync(dy, 0, 8 * (size_t)c->stride, c->stream));
  if (precond == NSG_PRECOND_IDENTITY)
    NSG_CUDA(cudaMemcpyAsync(dy, dx, 8 * (size_t)c->n_own, cudaMemcpyDeviceToDevice, c->stream));
  else {
    NSG_TRY(precond_initialize(c));
    NSG_TRY(precond_vmult(c, precond, dy, dx));
  }
  return get_vec(c, dy, y, c->n_own);
}

int nsg_ilu_apply(nsg_ctx *c, int32_t which, const double *x, double *y) {
  if (!c || !x || !y || which < 0 || which > 1) return fail(NSG_ERR_ARG, "bad argument");
  if (!c->have_mesh) return fail(NSG_ERR_STATE, "nsg_set_mesh first");
  NSG_CUDA(cudaSetDevice(c->device));
  NSG_TRY(precond_initialize(c));  // builds the blocks on first use
  CsrBlock &B = which == 0 ? c->blkA : c->blkM;
  double *dx = c->work, *dy = c->work + c->stride;
  NSG_TRY(put_vec(c, dx, x, B.n));
  NSG_TRY(ilu_apply(c, B, dy, dx));
  return get_vec(c, dy, y, B.n);
}

int nsg_boundary_force(nsg_ctx *c, int32_t boundary_id, double *out2) {
  if (!c || !out2) return fail(NSG_ERR_ARG, "null argument");
  if (!c->have_mesh) return fail(NSG_ERR_STATE, "nsg_set_mesh first");
  NSG_CUDA(cudaSetDevice(c->device));
  out2[0] = out2[1] = 0.0;
  double *fx = c->work + 2 * c->stride, *fy = c->work + 3 * c->stride;  // n_bfaces <= n_loc
  if (c->n_bfaces > c->stride) return fail(NSG_ERR_ARG, "more boundary faces than DoFs");
  if (c->n_bfaces > 0) {
    k_face_force<<<grid_for(c->n_bfaces, 128, 1 << 30), 128, 0, c->stream>>>(c->n_bfaces, boundary_id, c->n_own_u, c->bface_cell,
                                                                           c->bface_face, c->bface_tag, c->cell_vertices, c->cell_dofs,
                                                                           c->xy, c->geom, c->sol, c->prm.rho * c->prm.nu, fx, fy);
    NSG_LAUNCH_CHECK(c);
  }
  k_sum_ordered<<<1, 256, 0, c->stream>>>(c->n_bfaces, fx, fy, c->scal + 32);
  NSG_LAUNCH_CHECK(c);
  if (c->n_ranks > 1) NSG_NCCL(nccl_api().AllReduce(c->scal + 32, c->scal + 32, 2, ncclDouble, ncclSum, c->comm, c->stream));
  NSG_CUDA(cudaMemcpyAsync(out2, c->scal + 32, 16, cudaMemcpyDeviceToHost, c->stream));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  c->d2h += 16;
  return NSG_OK;
}

int nsg_set_cell_ownership(nsg_ctx *c, const int32_t *global_cell_id, const uint8_t *owned) {
  if (!c || !global_cell_id || !owned) return fail(NSG_ERR_ARG, "null argument");
  if (!c->have_mesh) return fail(NSG_ERR_STATE, "nsg_set_mesh first");
  for (int64_t i = 0; i < c->n_cells; ++i)
    if (global_cell_id[i] < 0 || global_cell_id[i] == PT_NONE) return fail(NSG_ERR_ARG, "global cell id out of range");
  NSG_CUDA(cudaSetDevice(c->device));
  dev_free(c->cell_gid), dev_free(c->cell_owned);
  NSG_TRY(upload(c, &c->cell_gid, global_cell_id, c->n_cells));
  NSG_TRY(upload(c, &c->cell_owned, owned, c->n_cells));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  return NSG_OK;
}

int nsg_eval_points(nsg_ctx *c, int64_t n, const double *xy, int32_t collective, double *values, double *grads, int64_t *cell) {
  if (!c || n < 0) return fail(NSG_ERR_ARG, "bad argument");
  if (!c->have_mesh) return fail(NSG_ERR_STATE, "nsg_set_mesh first");
  if (n == 0) return NSG_OK;
  if (!xy || !values) return fail(NSG_ERR_ARG, "null argument");
  NSG_CUDA(cudaSetDevice(c->device));
  if (!c->pidx.built) NSG_TRY(pt_build_index(c));
  NSG_TRY(pt_ensure_scratch(c, n, grads != nullptr));
  PointIndex &P = c->pidx;
  NSG_CUDA(cudaMemcpyAsync(P.pxy, xy, 16 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  NSG_TRY(pt_run(c, n, collective && c->n_ranks > 1 && c->comm, grads != nullptr));
  NSG_CUDA(cudaMemcpyAsync(values, P.vals, 24 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  if (grads) NSG_CUDA(cudaMemcpyAsync(grads, P.grads, 48 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  if (cell) NSG_CUDA(cudaMemcpyAsync(cell, P.cell, 8 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  NSG_CUDA(cudaStreamSynchronize(c->stream));
  P.last_n = n, P.last_grads = grads != nullptr;
  c->h2d += 16 * n;
  c->d2h += (24 + (grads ? 48 : 0) + (cell ? 8 : 0)) * n;
  return NSG_OK;
}

int nsg_points_index_info(nsg_ctx *c, double *out8) {
  if (!c || !out8) return fail(NSG_ERR_ARG, "null argument");
  const PointIndex &P = c->pidx;
  if (!P.built) return fail(NSG_ERR_STATE, "no point index yet: it is built by the first nsg_eval_points");
  const int64_t nb = (int64_t)P.grid.nx * P.grid.ny;
  out8[0] = P.grid.nx, out8[1] = P.grid.ny, out8[2] = P.h, out8[3] = (double)P.n_entries;
  out8[4] = (double)P.n_nonempty, out8[5] = P.max_bin, out8[6] = 8.0 * (nb + 1) + 4.0 * P.n_entries, out8[7] = P.build_ms;
  return NSG_OK;
}

int nsg_time_kernel(nsg_ctx *c, int32_t what, int32_t reps, double *ms_per_launch) {
  if (!c || !ms_per_launch || reps < 1) return fail(NSG_ERR_ARG, "bad argument");
  if (!c->have_mesh) return fail(NSG_ERR_STATE, "nsg_set_mesh first");
  NSG_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n_own;
  double *a = c->work + 2 * c->stride, *b = c->work + 3 * c->stride, *w = c->work + 4 * c->stride;
  NSG_CUDA(cudaMemsetAsync(c->scal, 0, 8, c->stream));
  if (what == 6 || what == 7) NSG_TRY(precond_initialize(c));  // factorise outside the timed region
  if (what == 8 && c->pidx.last_n == 0) return fail(NSG_ERR_STATE, "kernel 8 repeats the last nsg_eval_points: none yet");
  NSG_CUDA(cudaEventRecord(c->ev0, c->stream));
  for (int r = 0; r < reps; ++r) {
    switch (what) {
      case 8: NSG_TRY(pt_run(c, c->pidx.last_n, false, c->pidx.last_grads)); break;  // locate + evaluate, local mode
      case 6: NSG_TRY(ilu_apply(c, c->blkA, b, a)); break;            // ILU(0) apply of the velocity block (tuning key 4)
      case 7: NSG_TRY(ilu_apply(c, c->blkM, b + c->n_own_u, a + c->n_own_u)); break;  // ... of the pressure mass block
      case 0: NSG_TRY(launch_assembly(c)); break;
      case 1: NSG_TRY(dev_spmv(c, c->delta, a, nullptr)); break;
      case 2: NSG_TRY(dev_add_and_dot(c, n, a, c->scal, 1.0, b, w, c->scal + 1, nullptr)); break;
      case 3: NSG_TRY(dev_dot(c, n, a, b, c->scal + 1, nullptr)); break;
      case 4: NSG_TRY(halo_exchange(c, c->delta)); break;
      case 5: {  // FP64 pipe peak: sm_count x 16 CTAs x 256 threads x 8 chains x 2048 DFMA
        int sms = 0;
        NSG_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
        k_dfma_peak<<<sms * 16, DFMA_THREADS, 0, c->stream>>>(c->scal + 2, 0.999999, 1e-9);
        NSG_LAUNCH_CHECK(c);
        break;
      }
      default: return fail(NSG_ERR_ARG, "unknown kernel id");
    }
  }
  NSG_CUDA(cudaEventRecord(c->ev1, c->stream));
  NSG_CUDA(cudaEventSynchronize(c->ev1));
  float ms = 0;
  cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  *ms_per_launch = (double)ms / reps;
  if (what == 0) c->blocks_stale = true;
  return NSG_OK;
}

int nsg_set_tuning(nsg_ctx *c, int32_t key, int32_t value) {
  if (!c) return fail(NSG_ERR_ARG, "null context");
  switch (key) {
    case 0:
      if (value != 0 && value != 1 && value != 4 && value != 7) return fail(NSG_ERR_ARG, "spmv variant must be 0, 1, 4 or 7 (see nsg.h)");
      if (value == 7 && !c->have_paired) return fail(NSG_ERR_STATE, "the pattern has no node-pair structure");
      c->spmv_variant = value;
      for (auto &e : c->graphs) cudaGraphExecDestroy(e.exec);
      c->graphs.clear();  // captured segments embed the SpMV kernel
      return NSG_OK;
    case 2:
      c->use_graphs = value != 0;
      return NSG_OK;
    case 6:  // L2 prefetch distances of assembly variant 5, in chunks: records (low 16 bits), packets (high 16 bits); 0 = off
      if (value < 0) return fail(NSG_ERR_ARG, "prefetch distances must be >= 0");
      c->asm_pf_rec = value & 0xffff, c->asm_pf_pk = (value >> 16) & 0xffff;
      return NSG_OK;
    case 5:
      if (value < 0 || value > 2) return fail(NSG_ERR_ARG, "fused GMRES must be 0 (off), 1 (small systems) or 2 (whenever it fits)");
      c->gmres_fused = value;
      return NSG_OK;
    case 4:
      if (value < -1 || value > 2)
        return fail(NSG_ERR_ARG, "ILU solve variant must be -1 (choose per block), 0 (one launch per level), 1 (stamped single launch) or 2 (one CTA)");
      c->ilu_variant = value;
      return NSG_OK;
    case 3:
      if (value < 0 || value > 1) return fail(NSG_ERR_ARG, "orthogonalization must be 0 (modified) or 1 (classical Gram-Schmidt)");
      c->orthogonalization = value;
      for (auto &e : c->graphs) cudaGraphExecDestroy(e.exec);
      c->graphs.clear();
      return NSG_OK;
    case 1:
      if (value != 0 && value != 4 && value != 5) return fail(NSG_ERR_ARG, "assembly variant must be 0, 4 or 5 (see nsg.h)");
      if (value == 5 && c->have_mesh && !c->fan_ok)
        return fail(NSG_ERR_STATE, "the fan scheme (variant 5) cannot serve this mesh (not an oriented manifold triangulation with vertex valence <= 32)");
      if (value < 4) NSG_TRY(ensure_slot_worklists(c));
      if (value == 4) NSG_TRY(ensure_round_worklists(c, nullptr));
      if (value != c->asm_variant) c->p_rows_valid = false;
      c->asm_variant = value;
      return NSG_OK;
    default: return fail(NSG_ERR_ARG, "unknown tuning key");
  }
}

int nsg_get_counters(nsg_ctx *c, int64_t *launches, int64_t *h2d, int64_t *d2h) {
  if (!c) return fail(NSG_ERR_ARG, "null context");
  if (launches) *launches = c->launches;
  if (h2d) *h2d = c->h2d;
  if (d2h) *d2h = c->d2h;
  return NSG_OK;
}

int nsg_get_phase_ms(nsg_ctx *c, double *out3) {
  if (!c || !out3) return fail(NSG_ERR_ARG, "null argument");
  for (int i = 0; i < 3; ++i) out3[i] = c->phase_ms[i];
  return NSG_OK;
}

}  // extern "C"
