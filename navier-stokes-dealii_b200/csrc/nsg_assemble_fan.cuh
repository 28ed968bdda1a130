// nsg_assemble_fan.cuh — K1, "fan" scheme (assembly variant 5, the default): owner-computes assembly of the
// Jacobian, the pressure mass matrix and the residual (reference: src/NavierStokesSolver.cpp:203-347) with
// NO read-modify-write of the shared row image, NO commit rounds and NO table loads.
//
// Unit of work = one (row owner, cell) pair per lane, as in variant 4 (nsg_assemble.cuh).  What changes:
//  * Every pair is integrated in a ROTATED local frame of its cell in which the owner is local vertex 0
//    (vertex owners) or the midpoint of local edge 0 (edge owners).  The cyclic relabelling (v_r, v_r+1, v_r+2)
//    of a triangle is again a reference-element frame, so the owner's local index becomes a compile-time
//    constant (K = 0 or 3) and every pre-integrated table entry an immediate operand: no shared-memory tables.
//  * The integrals are written in barycentric form (grad lambda_j of the cell, nodal velocities): the second
//    Frechet term (cpp:265-269) needs 3 moments mu_j = sum_i u_i T_j[K][i] instead of a 7-point loop; the
//    velocity gradient at the vertices comes from the nodal values (cpp:229-233 restated for P2).  ~210 DFMA
//    per pair instead of ~380.
//  * The lanes of one owner sit in consecutive lanes of ONE warp, a vertex owner's cells in counter-clockwise
//    order around the vertex ("fan").  In a consistently oriented mesh the contribution of a cell to the
//    columns of its "previous" edge pairs with the "next"-edge contribution of the following cell of the fan:
//    one warp shuffle brings it over and the sum is stored ONCE.  The owner's own column (all cells of the fan)
//    is a segmented shuffle tree.  Hence every entry of the image is written exactly once, by a plain store:
//    no zero-fill, no loads from the image, no barriers between commit rounds.
//  * A streaming pre-pass writes one 192-byte packet per cell (nodal velocities, the cell's complete local
//    residual); grad lambda_j is static (geom8).  A lane loads only what no neighbouring lane holds: the values
//    of the nodes on the edge it shares with its predecessor in the fan come over by shuffle, the owner's own
//    value from the head lane, |det J| is recomputed from grad lambda.  6-7 instead of 17 16-byte loads per pair.
//    (Staging the packets in shared memory - cp.async, or one bulk copy per cell - was measured slower: 1.17 /
//    1.12 ms against 1.02 ms at 1.65 M cells, profiles/r02_summary.md; the chunk image leaves by one bulk copy.)
//  * The 2x2 blocks are stored with a lane-parity swizzle (odd lanes store the second column first): the column
//    offsets of velocity pairs are even, so unswizzled stores would use half of the banks per instruction.
// Summation order per entry is fixed (fan order), so the result is bitwise reproducible run to run; it differs
// from variant 4 / the reference's cell-loop order by rounding only (1e-16 relative).
// Meshes that are not consistently oriented, have an edge with more than two cells or a vertex with more than
// 32 cells are detected on the host and served by variant 4 (up to 32 cells per vertex) or else variant 0 (up to
// 64).  A pattern built on the device (nsg_set_pattern_from_cells) holds vertices of up to 34 cells inside the
// domain and 33 on the boundary.
#pragma once
#include "nsg_assemble.cuh"

namespace nsg {

#ifndef NSG_NPC6
#define NSG_NPC6 64
#endif
constexpr int NPC6 = NSG_NPC6;  // lanes (pairs) per CTA: two warps (measured: 64 lanes 0.943 ms, 128 lanes 0.965 ms, 256 lanes 1.099 ms at 1.65 M cells)
constexpr int PK6 = 24;    // doubles per cell packet: [0..11] nodal velocities u_i, [12..23] local residual of the 6 velocity nodes
constexpr int PK6S = 26;   // row stride of the pre-pass' transposition buffer (208 bytes: 16-byte aligned, conflict-free 128-bit stores)

// tables of the owner's row in the rotated frame, K = 0 (index 0) and K = 3 (index 1)
struct FanTab {
  double M[6];       // sum_q w psi_K psi_l
  double T[3][6];    // sum_q w lambda_j psi_K psi_i
  double K00[6], K01s[6], K11[6];
  double Bh[3][2];   // sum_q w dhat_c psi_K chi_m
};
__constant__ FanTab c_fan[2];
// pressure owner = rotated vertex 0: B[0][(b,l)] and Mp[0][n]
struct FanTabP {
  double Bp[6][2];  // sum_q w dhat_c psi_l chi_0
  double Mp[3];     // sum_q w chi_0 chi_n
};
__constant__ FanTabP c_fanp;

// geometry in barycentric form, once per mesh: [0..5] grad lambda_0, lambda_1, lambda_2; [6] |det J|; [7] 0
__global__ void k_cell_geometry8(int64_t T, const double *__restrict__ xy, const int32_t *__restrict__ cv, double *__restrict__ geom8) {
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= T) return;
  const int32_t v0 = cv[3 * c], v1 = cv[3 * c + 1], v2 = cv[3 * c + 2];
  const double x0 = xy[2 * v0], y0 = xy[2 * v0 + 1];
  const double J00 = xy[2 * v1] - x0, J01 = xy[2 * v2] - x0;
  const double J10 = xy[2 * v1 + 1] - y0, J11 = xy[2 * v2 + 1] - y0;
  const double det = J00 * J11 - J01 * J10;
  const double a00 = J11 / det, a01 = -J10 / det, a10 = -J01 / det, a11 = J00 / det;  // J^-T, as k_cell_geometry
  double2 *o = reinterpret_cast<double2 *>(geom8 + 8 * c);
  o[0] = make_double2(-(a00 + a01), -(a10 + a11));
  o[1] = make_double2(a00, a10);
  o[2] = make_double2(a01, a11);
  o[3] = make_double2(fabs(det), 0.0);
}

// ---- pre-pass: one 192-byte packet per cell ------------------------------------------------------------------
//   [0..11] nodal velocities u_i (FE_SimplexP(2) order: 3 vertices, 3 edges)
//   [12..23] the cell's complete local residual of its 6 velocity nodes (cpp:287-311)
// One thread per cell integrates; the packets of a CTA leave through shared memory, fully coalesced.
__global__ void __launch_bounds__(128, 4)
k_cell_packets6(int64_t T, const double *__restrict__ geom8, const int32_t *__restrict__ cell_dofs, const double *__restrict__ sol,
                const double *__restrict__ sol_old, const AsmParams P, double *__restrict__ cellpk) {
  __shared__ __align__(16) double s_out[128 * PK6S];
  const int t = threadIdx.x;
  const int64_t c0 = blockIdx.x * (int64_t)128;
  const int64_t c = c0 + t;
  double2 *mine = reinterpret_cast<double2 *>(s_out + t * PK6S);
  if (c < T) {
    const double2 *gp = reinterpret_cast<const double2 *>(geom8 + 8 * c);
    const double2 l0 = __ldg(gp), l1 = __ldg(gp + 1), l2 = __ldg(gp + 2), dd = __ldg(gp + 3);
    const double a00 = l1.x, a10 = l1.y, a01 = l2.x, a11 = l2.y, d = dd.x;
    (void)l0;
    const bool ns = !P.stokes;
    const double nurho = P.nu * P.rho, rd = P.rho * d, vd = nurho * d;
    double res[6][2];
#pragma unroll
    for (int k = 0; k < 6; ++k) res[k][0] = res[k][1] = 0.0;
    double u[6][2];
#pragma unroll
    for (int l = 0; l < 6; ++l) u[l][0] = u[l][1] = 0.0;
    if (ns) {
      const int32_t *cd = cell_dofs + 15 * c;
      double pr[3];
      int32_t dof[6];
#pragma unroll
      for (int l = 0; l < 6; ++l) {
        dof[l] = __ldg(cd + uidx(l));
        if ((dof[l] & 1) == 0) {  // owned velocity pairs start at an even index; ghost pairs need not (they follow the owned p)
          const double2 v = *reinterpret_cast<const double2 *>(sol + dof[l]);
          u[l][0] = v.x, u[l][1] = v.y;
        } else {
          u[l][0] = sol[dof[l]], u[l][1] = sol[dof[l] + 1];
        }
      }
#pragma unroll
      for (int m = 0; m < 3; ++m) pr[m] = sol[__ldg(cd + 3 * m + 2)];
      double h0[2][2] = {{0, 0}, {0, 0}}, hx[2][2] = {{0, 0}, {0, 0}}, hy[2][2] = {{0, 0}, {0, 0}};
#pragma unroll
      for (int l = 0; l < 6; ++l)
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int cc = 0; cc < 2; ++cc) {
            h0[a][cc] += u[l][a] * c_fe2.ga[l][cc];
            hx[a][cc] += u[l][a] * c_fe2.gb[l][cc];
            hy[a][cc] += u[l][a] * c_fe2.gc[l][cc];
          }
      double G0[2][2], Gx[2][2], Gy[2][2];
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        G0[a][0] = a00 * h0[a][0] + a01 * h0[a][1], G0[a][1] = a10 * h0[a][0] + a11 * h0[a][1];
        Gx[a][0] = a00 * hx[a][0] + a01 * hx[a][1], Gx[a][1] = a10 * hx[a][0] + a11 * hx[a][1];
        Gy[a][0] = a00 * hy[a][0] + a01 * hy[a][1], Gy[a][1] = a10 * hy[a][0] + a11 * hy[a][1];
      }
      // convective residual: cr[k][a] = sum_q w psi_k (U . grad) u_a   (cpp:297-301, index pattern of SURVEY F4)
      double cr[6][2];
#pragma unroll
      for (int k = 0; k < 6; ++k) cr[k][0] = cr[k][1] = 0.0;
#pragma unroll
      for (int q = 0; q < 7; ++q) {
        double U0 = 0, U1 = 0;
#pragma unroll
        for (int l = 0; l < 6; ++l) {
          U0 += u[l][0] * c_fe.psi[q][l];
          U1 += u[l][1] * c_fe.psi[q][l];
        }
        const double g00 = G0[0][0] + Gx[0][0] * c_fe2.qx[q] + Gy[0][0] * c_fe2.qy[q];
        const double g01 = G0[0][1] + Gx[0][1] * c_fe2.qx[q] + Gy[0][1] * c_fe2.qy[q];
        const double g10 = G0[1][0] + Gx[1][0] * c_fe2.qx[q] + Gy[1][0] * c_fe2.qy[q];
        const double g11 = G0[1][1] + Gx[1][1] * c_fe2.qx[q] + Gy[1][1] * c_fe2.qy[q];
        const double t0 = c_fe.w[q] * (U0 * g00 + U1 * g10), t1 = c_fe.w[q] * (U0 * g01 + U1 * g11);
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          cr[k][0] += c_fe.psi[q][k] * t0;
          cr[k][1] += c_fe.psi[q][k] * t1;
        }
      }
      const double S00 = a00 * a00 + a10 * a10, S01 = a00 * a01 + a10 * a11, S11 = a01 * a01 + a11 * a11;
      double du[6][2];
      if (P.use_mass) {
#pragma unroll
        for (int l = 0; l < 6; ++l) {
          if ((dof[l] & 1) == 0) {
            const double2 v = *reinterpret_cast<const double2 *>(sol_old + dof[l]);
            du[l][0] = u[l][0] - v.x, du[l][1] = u[l][1] - v.y;
          } else {
            du[l][0] = u[l][0] - sol_old[dof[l]], du[l][1] = u[l][1] - sol_old[dof[l] + 1];
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        double rv0 = 0, rv1 = 0, pb0 = 0, pb1 = 0;
#pragma unroll
        for (int l = 0; l < 6; ++l) {
          const double Kkl = S00 * c_fe2.K00[k][l] + S01 * c_fe2.K01s[k][l] + S11 * c_fe2.K11[k][l];
          rv0 += Kkl * u[l][0];
          rv1 += Kkl * u[l][1];
        }
#pragma unroll
        for (int m = 0; m < 3; ++m) {
          const double bh0 = c_fe2.Bh[k][m][0], bh1 = c_fe2.Bh[k][m][1];
          pb0 += pr[m] * (a00 * bh0 + a01 * bh1);
          pb1 += pr[m] * (a10 * bh0 + a11 * bh1);
        }
        double r0 = -vd * rv0 - rd * cr[k][0] + d * pb0, r1 = -vd * rv1 - rd * cr[k][1] + d * pb1;
        if (P.use_mass) {
          double t0 = 0, t1 = 0;
#pragma unroll
          for (int l = 0; l < 6; ++l) {
            t0 += c_fe2.Mh[k][l] * du[l][0];
            t1 += c_fe2.Mh[k][l] * du[l][1];
          }
          r0 -= P.rho * P.dt_inv * d * t0;
          r1 -= P.rho * P.dt_inv * d * t1;
        }
        res[k][0] = r0, res[k][1] = r1;
      }
    }
#pragma unroll
    for (int l = 0; l < 6; ++l) mine[l] = make_double2(u[l][0], u[l][1]);
#pragma unroll
    for (int k = 0; k < 6; ++k) mine[6 + k] = make_double2(res[k][0] + P.f0 * d * c_fe2.mh[k], res[k][1] + P.f1 * d * c_fe2.mh[k]);
  }
  __syncthreads();
  // coalesced write-out: 12 double2 per packet, consecutive threads -> consecutive 16-byte pieces
  const int64_t n_here = (T - c0 < 128) ? (T - c0) : 128;
  double2 *out = reinterpret_cast<double2 *>(cellpk + PK6 * c0);
  for (int i = t; i < (int)n_here * 12; i += 128) {
    const int cell = i / 12, part = i - 12 * cell;
    __stcs(out + i, *reinterpret_cast<const double2 *>(s_out + cell * PK6S + 2 * part));
  }
}

// ---- the owner's two rows of one cell in the rotated frame ---------------------------------------------------
// n1, n2 = grad lambda'_1, lambda'_2 (= columns of J'^-T), d = |det J|, u[0..5] = nodal velocities in rotated order.
// A[l] = {A00, A01, A10, A11} = entries [(a,K),(b,l)]; Bt[m] = {B^T[(0,K),m], B^T[(1,K),m]}.
template <int KT>
__device__ __forceinline__ void fan_rows(const double2 n1, const double2 n2, const double d, const double2 (&u)[6], const bool ns,
                                         const double mdt, const double nurho, const double rho, double (&A)[6][4], double (&Bt)[3][2]) {
  const FanTab &F = c_fan[KT];
  const double2 n0 = make_double2(-(n1.x + n2.x), -(n1.y + n2.y));
  const double S00 = n1.x * n1.x + n1.y * n1.y, S01 = n1.x * n2.x + n1.y * n2.y, S11 = n2.x * n2.x + n2.y * n2.y;
  const double md = mdt * d, vd = nurho * d, rd = rho * d;
#pragma unroll
  for (int l = 0; l < 6; ++l) {
    const double Kl = S00 * F.K00[l] + S01 * F.K01s[l] + S11 * F.K11[l];  // (1/d) sum_q w g_K.g_l   (cpp:252-257)
    const double D = md * F.M[l] + vd * Kl;                               // mass (cpp:249-251) + viscous
    A[l][0] = D, A[l][1] = 0.0, A[l][2] = 0.0, A[l][3] = D;
  }
  if (ns) {
    // rho d x velocity gradient at the three vertices: G^v_ab = sum_i u_i[a] (grad psi_i(v))_b
    const double2 e3m1 = make_double2(4.0 * u[3].x - u[1].x, 4.0 * u[3].y - u[1].y), e5m2 = make_double2(4.0 * u[5].x - u[2].x, 4.0 * u[5].y - u[2].y);
    const double2 e3m0 = make_double2(4.0 * u[3].x - u[0].x, 4.0 * u[3].y - u[0].y), e4m2 = make_double2(4.0 * u[4].x - u[2].x, 4.0 * u[4].y - u[2].y);
    const double2 e4m1 = make_double2(4.0 * u[4].x - u[1].x, 4.0 * u[4].y - u[1].y), e5m0 = make_double2(4.0 * u[5].x - u[0].x, 4.0 * u[5].y - u[0].y);
    const double2 N0 = make_double2(rd * n0.x, rd * n0.y), N1 = make_double2(rd * n1.x, rd * n1.y), N2 = make_double2(rd * n2.x, rd * n2.y);
    double G[3][4];
    {
      const double2 t0 = make_double2(3.0 * u[0].x, 3.0 * u[0].y), t1 = make_double2(3.0 * u[1].x, 3.0 * u[1].y), t2 = make_double2(3.0 * u[2].x, 3.0 * u[2].y);
      G[0][0] = t0.x * N0.x + e3m1.x * N1.x + e5m2.x * N2.x, G[0][1] = t0.x * N0.y + e3m1.x * N1.y + e5m2.x * N2.y;
      G[0][2] = t0.y * N0.x + e3m1.y * N1.x + e5m2.y * N2.x, G[0][3] = t0.y * N0.y + e3m1.y * N1.y + e5m2.y * N2.y;
      G[1][0] = t1.x * N1.x + e3m0.x * N0.x + e4m2.x * N2.x, G[1][1] = t1.x * N1.y + e3m0.x * N0.y + e4m2.x * N2.y;
      G[1][2] = t1.y * N1.x + e3m0.y * N0.x + e4m2.y * N2.x, G[1][3] = t1.y * N1.y + e3m0.y * N0.y + e4m2.y * N2.y;
      G[2][0] = t2.x * N2.x + e4m1.x * N1.x + e5m0.x * N0.x, G[2][1] = t2.x * N2.y + e4m1.x * N1.y + e5m0.x * N0.y;
      G[2][2] = t2.y * N2.x + e4m1.y * N1.x + e5m0.y * N0.x, G[2][3] = t2.y * N2.y + e4m1.y * N1.y + e5m0.y * N0.y;
    }
    // first Frechet term rho G_ab psi_K psi_l (cpp:259-263), G affine: sum_v G^v T[v][l]
#pragma unroll
    for (int l = 0; l < 6; ++l)
#pragma unroll
      for (int e = 0; e < 4; ++e) A[l][e] += G[0][e] * F.T[0][l] + G[1][e] * F.T[1][l] + G[2][e] * F.T[2][l];
    // second Frechet term rho psi_K U_b (g_l)_a (cpp:265-269): moments mu_j[b] = sum_q w psi_K U_b lambda_j
    double mu[3][2];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      double s0 = 0.0, s1 = 0.0;
#pragma unroll
      for (int i = 0; i < 6; ++i) s0 += u[i].x * F.T[j][i], s1 += u[i].y * F.T[j][i];
      mu[j][0] = s0, mu[j][1] = s1;
    }
    const double m00 = mu[0][0] + mu[1][0] + mu[2][0], m01 = mu[0][1] + mu[1][1] + mu[2][1];
    const double2 Nv[3] = {N0, N1, N2};
#pragma unroll
    for (int j = 0; j < 3; ++j) {  // vertex columns: grad psi_j = (4 lambda_j - 1) grad lambda_j
      const double c0 = 4.0 * mu[j][0] - m00, c1 = 4.0 * mu[j][1] - m01;
      A[j][0] += Nv[j].x * c0, A[j][1] += Nv[j].x * c1, A[j][2] += Nv[j].y * c0, A[j][3] += Nv[j].y * c1;
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {  // edge columns: grad psi_(3+j) = 4 (lambda_j grad lambda_j+1 + lambda_j+1 grad lambda_j)
      const int jn = (j + 1) % 3;
      const double2 Na = make_double2(4.0 * Nv[jn].x, 4.0 * Nv[jn].y), Nb = make_double2(4.0 * Nv[j].x, 4.0 * Nv[j].y);
      A[3 + j][0] += Na.x * mu[j][0] + Nb.x * mu[jn][0], A[3 + j][1] += Na.x * mu[j][1] + Nb.x * mu[jn][1];
      A[3 + j][2] += Na.y * mu[j][0] + Nb.y * mu[jn][0], A[3 + j][3] += Na.y * mu[j][1] + Nb.y * mu[jn][1];
    }
  }
  // B^T[(a,K),m] = -d sum_c (grad lambda'_(c+1))_a Bh[m][c]   (cpp:272-274)
#pragma unroll
  for (int m = 0; m < 3; ++m) {
    Bt[m][0] = -d * (n1.x * F.Bh[m][0] + n2.x * F.Bh[m][1]);
    Bt[m][1] = -d * (n1.y * F.Bh[m][0] + n2.y * F.Bh[m][1]);
  }
}

__device__ __forceinline__ double shfl_d(const double v, const int src) { return __shfl_sync(0xffffffffu, v, src); }

// Record of a lane (PairRec, 32 bytes):
//   cell    the cell (-1: idle lane)
//   k       canonical local index of the owner (3 bits) | partner lane in the warp << 3 (5) | has partner << 8 |
//           head << 9 (writes the owner's own column and residual) | write_next << 10 (the lane's "next"-side
//           columns have no partner: it stores them itself; = the lane has no predecessor in the fan) |
//           lanes of the owner after this one << 11 (5) | owner index in the chunk << 16 (8) |
//           predecessor lane << 24 (5; vertex owners: the lane whose "previous" edge is this lane's "next" edge)
//   off     [0..5] offsets of the column pairs of the ROTATED local nodes 0..5 in the owner's rows, [6..8] of the
//           three pressure columns (rotated order), [9] image offset of the owner's first row, [10] row length
// ChunkInfo: g0,g1 owners; rs, cnt image; pad != 0: the image has entries no lane writes (zero-fill first).
// what a lane loads for its pair (before the values its neighbours hold are shuffled in)
struct FanIn {
  double2 n1, n2, rk;  // grad lambda'_1, grad lambda'_2, the cell's local residual at the owner's node
  double2 u[6];        // nodal velocities in rotated order; [0], [1], [3] only where no neighbouring lane holds them
};
struct FanFlags {
  int kc, r, i1, i2, partner, pred, rem, gl;
  bool work, has_partner, head, write_next;
};
__device__ __forceinline__ FanFlags fan_flags(const uint4 ra) {
  FanFlags f;
  const uint32_t kw = ra.y;
  f.work = (int)ra.x >= 0;
  f.kc = (int)(kw & 7u), f.partner = (int)((kw >> 3) & 31u), f.rem = (int)((kw >> 11) & 31u), f.gl = (int)((kw >> 16) & 255u);
  f.pred = (int)((kw >> 24) & 31u);
  f.has_partner = (kw >> 8) & 1u, f.head = (kw >> 9) & 1u, f.write_next = (kw >> 10) & 1u;
  f.r = f.kc >= 3 ? f.kc - 3 : f.kc;
  f.i1 = f.r + 1 >= 3 ? f.r - 2 : f.r + 1, f.i2 = f.r + 2 >= 3 ? f.r - 1 : f.r + 2;
  return f;
}

// Everything after the loads: shuffle in what the neighbouring lanes hold, integrate the owner's two rows of the cell,
// combine the shared-edge contributions, store every entry of the image once.
__device__ __forceinline__ void fan_commit_u(const uint4 ra, const uint4 rb, const FanFlags f, const bool edge_owner, FanIn in,
                                             double *s_vals, double *s_res, const int lane, const AsmParams &P) {
  const bool work = f.work, head = f.head, write_next = f.write_next, has_partner = f.has_partner;
  const int partner = f.partner, pred = f.pred, rem = f.rem, gl = f.gl;
  double *row0 = s_vals + (rb.z >> 16), *row1 = row0 + (rb.w & 0xffffu);
  const uint32_t ow[5] = {ra.z, ra.w, rb.x, rb.y, rb.z};
  const bool ns = !P.stokes;
  const double mdt = (P.use_mass && ns) ? P.dt_inv : 0.0, nurho = P.nu * P.rho;
  double2 n1 = in.n1, n2 = in.n2, rk = in.rk;
  double2 u[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) u[i] = in.u[i];
  if (!work) {
    n1 = make_double2(1.0, 0.0), n2 = make_double2(0.0, 1.0), rk = make_double2(0.0, 0.0);
#pragma unroll
    for (int i = 0; i < 6; ++i) u[i] = make_double2(0.0, 0.0);
  }
  const double d = 1.0 / fabs(n1.x * n2.y - n1.y * n2.x);  // |det J| = 1 / |det (grad lambda'_1, grad lambda'_2)|
  if (!edge_owner) {
    // owner's own node from the head lane of the fan, the nodes of the "next" edge from the predecessor
    // (its vertex 2 is this lane's vertex 1, its edge 5 = (v2, v0) this lane's edge 3 = (v0, v1))
    const unsigned same = __match_any_sync(0xffffffffu, work ? gl : 256 + lane);
    const int hl = __ffs(same) - 1;
    const double h0x = shfl_d(u[0].x, hl), h0y = shfl_d(u[0].y, hl);
    const double p2x = shfl_d(u[2].x, pred), p2y = shfl_d(u[2].y, pred), p5x = shfl_d(u[5].x, pred), p5y = shfl_d(u[5].y, pred);
    if (!head) u[0] = make_double2(h0x, h0y);
    if (!write_next) u[1] = make_double2(p2x, p2y), u[3] = make_double2(p5x, p5y);
  } else {
    // the other cell of the edge runs it the other way round: its vertex 0 is this lane's vertex 1; the owner's own
    // node (3) is loaded by the head lane only
    const double q0x = shfl_d(u[0].x, partner), q0y = shfl_d(u[0].y, partner), q3x = shfl_d(u[3].x, partner), q3y = shfl_d(u[3].y, partner);
    if (has_partner) u[1] = make_double2(q0x, q0y);
    if (!head) u[3] = make_double2(q3x, q3y);
  }
  double A[6][4], Bt[3][2];
  if (!edge_owner)
    fan_rows<0>(n1, n2, d, u, ns, mdt, nurho, P.rho, A, Bt);
  else
    fan_rows<1>(n1, n2, d, u, ns, mdt, nurho, P.rho, A, Bt);
  if (!work) {
#pragma unroll
    for (int l = 0; l < 6; ++l) A[l][0] = A[l][1] = A[l][2] = A[l][3] = 0.0;
#pragma unroll
    for (int m = 0; m < 3; ++m) Bt[m][0] = Bt[m][1] = 0.0;
  }
  auto off = [&](int l) -> int { return (int)((ow[l >> 1] >> ((l & 1) * 16)) & 0xffffu); };
  // the column offsets of velocity pairs are even: odd lanes store the second column first, so that one store
  // instruction of the warp spreads over all banks
  const int sw = lane & 1;
  auto st_block = [&](int l, double v0, double v1, double v2, double v3) {
    const int o = off(l);
    row0[o + sw] = sw ? v1 : v0, row1[o + sw] = sw ? v3 : v2;
    row0[o + 1 - sw] = sw ? v0 : v1, row1[o + 1 - sw] = sw ? v2 : v3;
  };
  auto st_p = [&](int m, double v0, double v1) {
    const int o = off(6 + m);
    row0[o] = v0, row1[o] = v1;
  };
  if (!edge_owner) {
    // -- vertex owner: the lane's "previous"-edge columns (vertex 2, midpoint 5, pressure 2) take the "next"-edge
    //    contribution (vertex 1, midpoint 3, pressure 1) of the following cell of the fan
    double x1[4], x3[4], xb[2];
#pragma unroll
    for (int e = 0; e < 4; ++e) x1[e] = shfl_d(A[1][e], partner), x3[e] = shfl_d(A[3][e], partner);
    xb[0] = shfl_d(Bt[1][0], partner), xb[1] = shfl_d(Bt[1][1], partner);
    if (!has_partner) {
#pragma unroll
      for (int e = 0; e < 4; ++e) x1[e] = x3[e] = 0.0;
      xb[0] = xb[1] = 0.0;
    }
    // the owner's own column, pressure column and residual: segmented tree over the owner's lanes
    double sv[8] = {A[0][0], A[0][1], A[0][2], A[0][3], Bt[0][0], Bt[0][1], rk.x, rk.y};
    const int maxrem = __reduce_max_sync(0xffffffffu, work ? rem : 0);
    for (int dlt = 1; dlt <= maxrem; dlt <<= 1) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const double o = __shfl_down_sync(0xffffffffu, sv[e], dlt);
        if (dlt <= rem) sv[e] += o;
      }
    }
    if (work) {
      st_block(2, A[2][0] + x1[0], A[2][1] + x1[1], A[2][2] + x1[2], A[2][3] + x1[3]);
      st_block(5, A[5][0] + x3[0], A[5][1] + x3[1], A[5][2] + x3[2], A[5][3] + x3[3]);
      st_p(2, Bt[2][0] + xb[0], Bt[2][1] + xb[1]);
      st_block(4, A[4][0], A[4][1], A[4][2], A[4][3]);
      if (write_next) {
        st_block(1, A[1][0], A[1][1], A[1][2], A[1][3]);
        st_block(3, A[3][0], A[3][1], A[3][2], A[3][3]);
        st_p(1, Bt[1][0], Bt[1][1]);
      }
      if (head) {
        st_block(0, sv[0], sv[1], sv[2], sv[3]);
        st_p(0, sv[4], sv[5]);
        s_res[2 * gl] = sv[6], s_res[2 * gl + 1] = sv[7];
      }
    }
  } else {
    // -- edge owner (midpoint of rotated edge 0 = v0 v1): my column of v0 takes the partner's column of ITS v1; the
    //    head lane also sums the owner's own column (node 3) and the residual
    double x1[4], x3[4], xb[2], xr[2];
#pragma unroll
    for (int e = 0; e < 4; ++e) x1[e] = shfl_d(A[1][e], partner), x3[e] = shfl_d(A[3][e], partner);
    xb[0] = shfl_d(Bt[1][0], partner), xb[1] = shfl_d(Bt[1][1], partner);
    xr[0] = shfl_d(rk.x, partner), xr[1] = shfl_d(rk.y, partner);
    if (!has_partner) {
#pragma unroll
      for (int e = 0; e < 4; ++e) x1[e] = x3[e] = 0.0;
      xb[0] = xb[1] = xr[0] = xr[1] = 0.0;
    }
    if (work) {
      st_block(0, A[0][0] + x1[0], A[0][1] + x1[1], A[0][2] + x1[2], A[0][3] + x1[3]);
      st_p(0, Bt[0][0] + xb[0], Bt[0][1] + xb[1]);
      st_block(2, A[2][0], A[2][1], A[2][2], A[2][3]);
      st_block(4, A[4][0], A[4][1], A[4][2], A[4][3]);
      st_block(5, A[5][0], A[5][1], A[5][2], A[5][3]);
      st_p(2, Bt[2][0], Bt[2][1]);
      if (write_next) {
        st_block(1, A[1][0], A[1][1], A[1][2], A[1][3]);
        st_p(1, Bt[1][0], Bt[1][1]);
      }
      if (head) {
        st_block(3, A[3][0] + x3[0], A[3][1] + x3[1], A[3][2] + x3[2], A[3][3] + x3[3]);
        s_res[2 * gl] = rk.x + xr[0], s_res[2 * gl + 1] = rk.y + xr[1];
      }
    }
  }
}

template <int MINB>
__global__ void __launch_bounds__(NPC6, (MINB * 128) / NPC6)
k_assemble_u6(const WorkList wl, double *__restrict__ vals, double *__restrict__ R, const double *__restrict__ cellpk,
              const double *__restrict__ geom8, const AsmParams P, const int pf_rec, const int pf_pk) {
  extern __shared__ __align__(16) double s_vals[];
  const int t = threadIdx.x, lane = t & 31;
  const int64_t b = blockIdx.x;
  const uint4 *rp = reinterpret_cast<const uint4 *>(wl.recs + b * NPC6 + t);
  const uint4 ra = __ldcs(rp), rb = __ldcs(rp + 1);
  const ChunkInfo ci = wl.chunks[b];
  // Pull the lines of chunks that will run a little later towards L2: the record of chunk b + pf_rec (one sector per
  // lane, no register held), and - through the cell id of chunk b + pf_pk's record - its packet and geometry lines.
  if (pf_rec > 0 && b + pf_rec < wl.n_chunks) pf_l2(wl.recs + (b + pf_rec) * NPC6 + t);
  int pf_cell = -1;
  if (pf_pk > 0 && b + pf_pk < wl.n_chunks) pf_cell = __ldg(&wl.recs[(b + pf_pk) * NPC6 + t].cell);
  const int cnt = ci.cnt, ng = ci.g1 - ci.g0;
  double *s_res = s_vals + cnt;
  if (ci.pad) {  // the pattern has entries no cell contributes to: they must read zero
    const int n2 = (cnt + 2 * ng + 1) >> 1;
    double2 *z = reinterpret_cast<double2 *>(s_vals);
    for (int i = t; i < n2; i += NPC6) z[i] = make_double2(0.0, 0.0);
    __syncthreads();
  }
  const FanFlags f = fan_flags(ra);
  // uniform over the warp: the host packs vertex owners and edge owners into different warps (idle padding lanes have no
  // type of their own and must take the branch of their warp: the shuffles are full-mask)
  const bool edge_owner = __any_sync(0xffffffffu, f.work && f.kc >= 3);
  const int64_t cell = f.work ? (int)ra.x : 0;
  const double2 *gp = reinterpret_cast<const double2 *>(geom8 + 8 * cell);
  const double2 *pk = reinterpret_cast<const double2 *>(cellpk + PK6 * cell);
  FanIn in;
  in.n1 = in.n2 = in.rk = make_double2(0.0, 0.0);
#pragma unroll
  for (int i = 0; i < 6; ++i) in.u[i] = make_double2(0.0, 0.0);
  if (f.work) {  // everything a neighbouring lane does not hold
    in.n1 = __ldg(gp + f.i1), in.n2 = __ldg(gp + f.i2);
    in.u[2] = __ldg(pk + f.i2), in.u[4] = __ldg(pk + 3 + f.i1), in.u[5] = __ldg(pk + 3 + f.i2);
    in.rk = __ldg(pk + 6 + f.kc);
    if (!edge_owner) {
      if (f.head) in.u[0] = __ldg(pk + f.r);
      if (f.write_next) in.u[1] = __ldg(pk + f.i1), in.u[3] = __ldg(pk + 3 + f.r);  // no predecessor to take them from
    } else {
      in.u[0] = __ldg(pk + f.r);
      if (f.head) in.u[3] = __ldg(pk + 3 + f.r);
      if (!f.has_partner) in.u[1] = __ldg(pk + f.i1);
    }
  }
  if (pf_cell >= 0) {
    const char *q = reinterpret_cast<const char *>(cellpk + PK6 * (int64_t)pf_cell);
    pf_l2(q), pf_l2(q + 128), pf_l2(geom8 + 8 * (int64_t)pf_cell);
  }
  fan_commit_u(ra, rb, f, edge_owner, in, s_vals, s_res, lane, P);
  __syncthreads();
  double *out = vals + ci.rs;
  if (((ci.rs | (int64_t)cnt) & 1) == 0) {
    if (t == 0 && cnt > 0) bulk_store_image(out, s_vals, (uint32_t)cnt * 8u);
  } else {
    for (int i = t; i < cnt; i += NPC6) __stcs(out + i, s_vals[i]);
  }
  for (int i = t; i < 2 * ng; i += NPC6) R[2 * (int64_t)ci.g0 + i] = s_res[i];
}

// (A persistent, software-pipelined form of this kernel - next chunk's values copied into lane-private shared-memory
//  slots by cp.async while the current chunk is integrated, records and headers one and two chunks ahead in registers,
//  two image buffers so that the TMA write-out of chunk i overlaps chunk i+1 - was built and measured in round 2:
//  bitwise the same result, long_scoreboard stalls 4.3 -> 1.2 per issue, but the SAME time (0.964 vs 0.957 ms at
//  1.65 M cells, 10.93 vs 10.78 ms at 18.9 M): with ~1050 issued instructions per warp and chunk, two thirds of them
//  shuffles, selects and address arithmetic, the kernel is bound by instruction issue at 12-16 warps per SM, not by
//  the loads.  It was not kept; profiles/r02_summary.md has the numbers.)

// ---- pressure rows (B, the structurally present zero p-p block, pressure mass): vertex fans only --------------
// Record as above; off[0..5] = column pairs of the rotated P2 nodes in the Jacobian row, off[6..8] = the three
// pressure columns in the pressure-mass row, off[9] = image offset of the Jacobian row, off[10] = offset of the
// pressure-mass row in the mass image.  The p-p block of the Jacobian is never written: the image is zero-filled.
// Reads the geometry and nu only, so launch_assembly runs it once and again only after nu, the assembly variant or a
// Dirichlet constraint on a pressure row changed what it writes (nsg_ctx::p_rows_valid).
__global__ void __launch_bounds__(NPC6, (6 * 128) / NPC6)
k_assemble_p6(const WorkList wl, int64_t n_own_u, double *__restrict__ vals, double *__restrict__ pm_vals, double *__restrict__ R,
              const double *__restrict__ geom8, const AsmParams P) {
  extern __shared__ __align__(16) double s_mem[];
  const int t = threadIdx.x;
  const int64_t b = blockIdx.x;
  const uint4 *rp = reinterpret_cast<const uint4 *>(wl.recs + b * NPC6 + t);
  const uint4 ra = __ldcs(rp), rb = __ldcs(rp + 1);
  const ChunkInfo ci = wl.chunks[b];
  const bool work = (int)ra.x >= 0;
  const uint32_t kw = ra.y;
  const int kc = (int)(kw & 7u), partner = (int)((kw >> 3) & 31u), rem = (int)((kw >> 11) & 31u);
  const bool has_partner = (kw >> 8) & 1u, head = (kw >> 9) & 1u, write_next = (kw >> 10) & 1u;
  const int r = kc;
  const int i1 = r + 1 >= 3 ? r - 2 : r + 1, i2 = r + 2 >= 3 ? r - 1 : r + 2;
  double2 n1 = make_double2(0, 0), n2 = n1, dd = n1;
  if (work) {
    const double2 *gp = reinterpret_cast<const double2 *>(geom8 + 8 * (int64_t)(int)ra.x);
    n1 = __ldg(gp + i1), n2 = __ldg(gp + i2), dd = __ldg(gp + 3);
  }
  const int cnt = ci.cnt, mcnt = ci.mcnt, ng = ci.g1 - ci.g0;
  double *s_vals = s_mem, *s_pm = s_mem + cnt;
  {
    const int n2z = (cnt + mcnt + 1) >> 1;
    double2 *z = reinterpret_cast<double2 *>(s_vals);
    for (int i = t; i < n2z; i += NPC6) z[i] = make_double2(0.0, 0.0);
  }
  __syncthreads();
  double *row = s_vals + (rb.z >> 16), *mrow = s_pm + (rb.w & 0xffffu);
  const uint32_t ow[5] = {ra.z, ra.w, rb.x, rb.y, rb.z};
  auto off = [&](int l) -> int { return (int)((ow[l >> 1] >> ((l & 1) * 16)) & 0xffffu); };
  const double d = dd.x, dnu = d / P.nu;
  double Bx[6], By[6], M[3];
#pragma unroll
  for (int l = 0; l < 6; ++l) {  // B[0][(b,l)] = -d sum_c (grad lambda'_(c+1))_b Bp[l][c]   (cpp:277-279)
    Bx[l] = work ? -d * (n1.x * c_fanp.Bp[l][0] + n2.x * c_fanp.Bp[l][1]) : 0.0;
    By[l] = work ? -d * (n1.y * c_fanp.Bp[l][0] + n2.y * c_fanp.Bp[l][1]) : 0.0;
  }
#pragma unroll
  for (int n = 0; n < 3; ++n) M[n] = work ? c_fanp.Mp[n] * dnu : 0.0;  // cpp:282-284
  double x1[2], x3[2], xm;
  x1[0] = shfl_d(Bx[1], partner), x1[1] = shfl_d(By[1], partner);
  x3[0] = shfl_d(Bx[3], partner), x3[1] = shfl_d(By[3], partner);
  xm = shfl_d(M[1], partner);
  if (!has_partner) x1[0] = x1[1] = x3[0] = x3[1] = xm = 0.0;
  double sv[3] = {Bx[0], By[0], M[0]};
  const int maxrem = __reduce_max_sync(0xffffffffu, work ? rem : 0);
  for (int dlt = 1; dlt <= maxrem; dlt <<= 1) {
#pragma unroll
    for (int e = 0; e < 3; ++e) {
      const double o = __shfl_down_sync(0xffffffffu, sv[e], dlt);
      if (dlt <= rem) sv[e] += o;
    }
  }
  const int sw = t & 1;  // lane-parity swizzle, as in k_assemble_u6
  auto st_pair = [&](int l, double v0, double v1) {
    const int o = off(l);
    row[o + sw] = sw ? v1 : v0;
    row[o + 1 - sw] = sw ? v0 : v1;
  };
  if (work) {
    st_pair(2, Bx[2] + x1[0], By[2] + x1[1]);
    st_pair(5, Bx[5] + x3[0], By[5] + x3[1]);
    st_pair(4, Bx[4], By[4]);
    mrow[off(8)] = M[2] + xm;
    if (write_next) {
      st_pair(1, Bx[1], By[1]);
      st_pair(3, Bx[3], By[3]);
      mrow[off(7)] = M[1];
    }
    if (head) {
      st_pair(0, sv[0], sv[1]);
      mrow[off(6)] = sv[2];
    }
  }
  __syncthreads();
  double *out = vals + ci.rs, *mout = pm_vals + ci.ms;
  for (int i = t; i < cnt; i += NPC6) __stcs(out + i, s_vals[i]);
  for (int i = t; i < mcnt; i += NPC6) __stcs(mout + i, s_pm[i]);
  // no statement of the reference tests the pressure space: R_p == 0 (SURVEY F4)
  for (int i = t; i < ng; i += NPC6) R[n_own_u + ci.g0 + i] = 0.0;
}

}  // namespace nsg
