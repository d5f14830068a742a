// element_p1tet.cuh -- factorised P1-P1 tetrahedron kernels for the G-metric SUPG/PSPG/LSIC form
// (NavierStokes/NavierStokesChannelFlow.py:220-251), the flagship element pair of the hot path.
//
// Unit of work: one (vertex, incident cell) INCIDENCE.  The cell's vertices are passed with the row vertex
// FIRST (the caller rotates them), so everything below indexes statically.  The function returns the four
// 4x4 blocks of the element Jacobian whose rows belong to that vertex -- rows = (u_x, u_y, u_z, p) test
// functions of vertex 0, columns = (u_x, u_y, u_z, p) trial functions of vertex n, n = 0..3 -- and the
// matching four residual entries.
//
// Algebra (SURVEY.md Appendix A.3/A.7, re-derived in DESIGN.md): with P1 functions every gradient is a cell
// constant, and the degree-2 rule has one point per vertex with N_n(q) = a + e [q == n], e = b - a.  Hence
//   sum_q N_n(q) f_q = a sum_q f_q + e f_n :
// every quadrature sum splits into a cell total plus the value at the point attached to the column vertex.
// Only tau_q (one rsqrt per point) is genuinely nonlinear.
#pragma once
#include "element_generic.cuh"

namespace nsgpu {

#if defined(__CUDA_ARCH__)
#define NS_RSQRT(x) rsqrt(x)
#else
#define NS_RSQRT(x) (1.0 / sqrt(x))
#endif

constexpr double P1T_A = 0.1381966011250105;   // (5 - sqrt 5) / 20
constexpr double P1T_E = 0.4472135954999579;   // b - a = sqrt(5) / 5

// x: 4 vertices x 3 coordinates, u: 4 x 3 nodal velocities, p: 4 nodal pressures; vertex 0 = row vertex.
// The metric tensor G = K^T K = sum over the three NON-ORIGIN vertices of g_k (x) g_k is the one quantity of the
// form that depends on which vertex dolfinx lists first, so the caller says where the cell's original
// vertex 0 sits after the rotation: position 0 (row_is_origin) or position 1.
// blk[n][4*r + d]: row r (0..2 velocity component, 3 pressure) of vertex 0, column d of vertex n.
// fr[r]: residual entries of vertex 0.  Un-zeroed (Dirichlet handling is the caller's).
template <bool WANT_J, bool WANT_F>
NS_HD void p1tet_rowslab(const FormParams& fp, const bool row_is_origin, const double (&x)[4][3], const double (&u)[4][3],
                         const double (&p)[4], double (&blk)[4][16], double (&fr)[4]) {
  // ---- geometry: K = J^-1, gradients g_n, |det J| ----
  double J[3][3];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) J[i][j] = x[j + 1][i] - x[0][i];
  const double c00 = J[1][1] * J[2][2] - J[1][2] * J[2][1];
  const double c01 = J[1][2] * J[2][0] - J[1][0] * J[2][2];
  const double c02 = J[1][0] * J[2][1] - J[1][1] * J[2][0];
  const double det = J[0][0] * c00 + J[0][1] * c01 + J[0][2] * c02;
  const double idet = 1.0 / det;
  double g[4][3];  // g[n][j] = d phi_n / d x_j ; g[k+1][j] = K[k][j]
  g[1][0] = c00 * idet; g[2][0] = c01 * idet; g[3][0] = c02 * idet;
  g[1][1] = (J[0][2] * J[2][1] - J[0][1] * J[2][2]) * idet;
  g[2][1] = (J[0][0] * J[2][2] - J[0][2] * J[2][0]) * idet;
  g[3][1] = (J[0][1] * J[2][0] - J[0][0] * J[2][1]) * idet;
  g[1][2] = (J[0][1] * J[1][2] - J[0][2] * J[1][1]) * idet;
  g[2][2] = (J[0][2] * J[1][0] - J[0][0] * J[1][2]) * idet;
  g[3][2] = (J[0][0] * J[1][1] - J[0][1] * J[1][0]) * idet;
#pragma unroll
  for (int j = 0; j < 3; ++j) g[0][j] = -(g[1][j] + g[2][j] + g[3][j]);
  const double W = fabs(det) * (1.0 / 24.0);   // weight of every point; cell volume V = 4 W
  const double V = 4.0 * W;

  // metric tensor G = K^T K (symmetric), tr G, G:G
  double G[3][3], gk[3];   // gk: gradient of the non-origin vertex among rotated positions 0 / 1
#pragma unroll
  for (int j = 0; j < 3; ++j) gk[j] = row_is_origin ? g[1][j] : g[0][j];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = i; j < 3; ++j) {
      G[i][j] = gk[i] * gk[j] + g[2][i] * g[2][j] + g[3][i] * g[3][j];
      G[j][i] = G[i][j];
    }
  const double trG = G[0][0] + G[1][1] + G[2][2];
  const double GG = G[0][0] * G[0][0] + G[1][1] * G[1][1] + G[2][2] * G[2][2] +
                    2.0 * (G[0][1] * G[0][1] + G[0][2] * G[0][2] + G[1][2] * G[1][2]);
  const double Cst = fp.Ci * fp.nu * fp.nu * GG;
  const double itrG = 1.0 / trG;

  // ---- cell-constant fields: D = grad u (D[i][j] = d_j u_i), P = grad p, div u ----
  double D[3][3], P[3], U[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    U[i] = u[0][i] + u[1][i] + u[2][i] + u[3][i];
#pragma unroll
    for (int j = 0; j < 3; ++j) D[i][j] = u[0][i] * g[0][j] + u[1][i] * g[1][j] + u[2][i] * g[2][j] + u[3][i] * g[3][j];
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) P[j] = p[0] * g[0][j] + p[1] * g[1][j] + p[2] * g[2][j] + p[3] * g[3][j];
  const double divu = D[0][0] + D[1][1] + D[2][2];

  // ---- the four quadrature points (point q sits next to vertex q) ----
  double uq[4][3], Guq[4][3], wt[4], al[4], be[4];   // wt = W tau, al = W tau a_0(q), be = W tau^3 a_0(q)
  double s[3] = {0, 0, 0}, Q[6] = {0, 0, 0, 0, 0, 0}, ZG[3] = {0, 0, 0}, TR[3] = {0, 0, 0};
  double tbar = 0.0, nuLbar = 0.0;
  double Y1[3][3], Y3[3] = {0, 0, 0};   // Y1[d][c] = sum_q be_q (Gu_q)_d u_q,c ; Y3[d] = sum_q be_q (Gu_q)_d
#pragma unroll
  for (int d = 0; d < 3; ++d)
#pragma unroll
    for (int c = 0; c < 3; ++c) Y1[d][c] = 0.0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    double arg = Cst, r[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) uq[q][i] = P1T_A * U[i] + P1T_E * u[q][i];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      Guq[q][i] = G[i][0] * uq[q][0] + G[i][1] * uq[q][1] + G[i][2] * uq[q][2];
      arg += uq[q][i] * Guq[q][i];
    }
    const double tau = NS_RSQRT(arg);             // tau_SUPS (:238)
    const double wtau = W * tau;
    nuLbar += wtau * arg;                          // W nu_L = W sqrt(arg) / trG = W tau arg / trG (scaled below)
    // r = dot(u, grad u) + grad p  (res_M for P1: -div sigma = grad p)
#pragma unroll
    for (int j = 0; j < 3; ++j) r[j] = P[j] + uq[q][0] * D[0][j] + uq[q][1] * D[1][j] + uq[q][2] * D[2][j];
    const double a0 = r[0] * g[0][0] + r[1] * g[0][1] + r[2] * g[0][2];   // a_m(q) = r_q . g_m, m = row vertex
    wt[q] = wtau;
    al[q] = wtau * a0;
    be[q] = al[q] * tau * tau;
    tbar += wtau;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double wu = wtau * uq[q][i];
      s[i] += wu;
      ZG[i] += wtau * Guq[q][i];
      TR[i] += wtau * r[i];
      Y3[i] += be[q] * Guq[q][i];
    }
    Q[0] += wtau * uq[q][0] * uq[q][0]; Q[1] += wtau * uq[q][0] * uq[q][1]; Q[2] += wtau * uq[q][0] * uq[q][2];
    Q[3] += wtau * uq[q][1] * uq[q][1]; Q[4] += wtau * uq[q][1] * uq[q][2]; Q[5] += wtau * uq[q][2] * uq[q][2];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const double bg = be[q] * Guq[q][d];
#pragma unroll
      for (int c = 0; c < 3; ++c) Y1[d][c] += bg * uq[q][c];
    }
  }
  nuLbar *= itrG;
  const double Qm[3][3] = {{Q[0], Q[1], Q[2]}, {Q[1], Q[3], Q[4]}, {Q[2], Q[4], Q[5]}};

  // ---- row-vertex (m = 0) constants ----
  double H[3], ub[3], Dub[3];   // H[d] = (D g_0)_d ; ub = sum_q W N_0(q) u_q ; Dub = D ub
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    H[d] = D[d][0] * g[0][0] + D[d][1] * g[0][1] + D[d][2] * g[0][2];
    ub[d] = W * (P1T_A * U[d] + P1T_E * uq[0][d]);
  }
  const double TR0 = TR[0] * g[0][0] + TR[1] * g[0][1] + TR[2] * g[0][2];   // (sum_q W tau r_q) . g_0

  if (WANT_F) {
    const double pbarV = W * (p[0] + p[1] + p[2] + p[3]);                    // sum_q W p_q
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      Dub[c] = D[c][0] * ub[0] + D[c][1] * ub[1] + D[c][2] * ub[2];          // Galerkin convection
      const double supg = al[0] * uq[0][c] + al[1] * uq[1][c] + al[2] * uq[2][c] + al[3] * uq[3][c];
      fr[c] = Dub[c] + fp.nu * V * H[c] - pbarV * g[0][c] + supg + nuLbar * divu * g[0][c];
    }
    fr[3] = W * divu + TR0;                                                   // q div u + tau r . grad q
  }

  if (WANT_J) {
    const double kap = divu * itrG;
    const double M_off = W * (4.0 * P1T_A * P1T_A + 2.0 * P1T_A * P1T_E);    // sum_q W N_m N_n, m != n
    const double M_dia = M_off + W * P1T_E * P1T_E;
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      const double L = g[0][0] * g[n][0] + g[0][1] * g[n][1] + g[0][2] * g[n][2];
      const double Mmn = (n == 0) ? M_dia : M_off;
      // point-n parts of the N_n-weighted sums
      const double ebn = P1T_E * be[n], ewn = P1T_E * wt[n];
      double Sn[3], Zn[3], X3[3];
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        Sn[d] = P1T_A * s[d] + ewn * uq[n][d];                                // S[c,n] = sum_q W tau u_c N_n
        Zn[d] = (P1T_A * ZG[d] + ewn * Guq[n][d]) * kap;                      // Z[d,n] div u / tr G
        X3[d] = P1T_A * Y3[d] + ebn * Guq[n][d];                              // sum_q W tau^3 N_n (Gu)_d a_m
      }
      const double tn = P1T_A * tbar + ewn;                                    // sum_q W tau N_n
      const double X2 = P1T_A * TR0 + P1T_E * al[n];                           // sum_q W tau N_n a_m
      const double ubgn = ub[0] * g[n][0] + ub[1] * g[n][1] + ub[2] * g[n][2];
      const double dia = ubgn + fp.nu * V * L + X2;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          double v = Mmn * D[c][d];
          v -= P1T_A * Y1[d][c] + ebn * Guq[n][d] * uq[n][c];
          v += Sn[c] * H[d] + Qm[c][d] * L + Zn[d] * g[0][c] + nuLbar * g[0][c] * g[n][d];
          if (c == d) v += dia;
          blk[n][4 * c + d] = v;
        }
        blk[n][4 * c + 3] = s[c] * L - W * g[0][c];                           // A_vp
      }
#pragma unroll
      for (int d = 0; d < 3; ++d) blk[n][12 + d] = W * g[n][d] - X3[d] + tn * H[d] + s[d] * L;   // A_pv
      blk[n][15] = tbar * L;                                                   // A_pp
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// Register-lean version of p1tet_rowslab (what the CUDA kernel runs).  Same algebra, reorganised so that
//   * everything that does not depend on the column vertex n is folded once into C0 (3x3), P0 (3) and a few scalars:
//       A_vv[c][d] = C0[c][d] + [n == 0] e^2 W D[c][d] + L Q[c][d] + uq_n[c] t1[d] + g_0[c] t2[d] + delta_cd dia
//       A_pv[d]    = P0[d] + W g_n[d] + t1[d] + s[d] L
//     with t1 = e W tau_n (H - tau_n^2 a_0(n) Gu_n),  t2 = e W tau_n kappa Gu_n + nuL g_n   (per block: ~70 FMA);
//   * the per-point data of points 1..3 is parked by `scratch` (the warp-specialised kernel uses the thread's lane of
//     tensor memory, the other kernels its own, not yet written, staging slots in shared memory) and fetched back right
//     before the block that needs it;
//   * each finished 4x4 block is handed to `emit(n, blk)` immediately (Dirichlet handling + staging store), the first one
//     after `scratch.before_first_emit()`.
// Live state during the block loop is ~55 doubles instead of ~100, which gives ptxas room to interleave the
// independent FMA chains (the fp64 pipe needs ILP >= 2 at 8 warps/SM: tools/microbench.cu).
struct P1TetPoint { double uq[3], Gu[3], ew, eb, ea; };   // ew = e W tau, eb = e W tau^3 a_0, ea = e W tau a_0

template <bool WANT_J, bool WANT_F, class Scratch, class Emit>
NS_HD void p1tet_rowslab2(const FormParams& fp, const bool row_is_origin, const double (&x)[4][3], const double (&u)[4][3],
                          const double (&p)[4], double (&fr)[4], Scratch&& scratch, Emit&& emit) {
  double J[3][3];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) J[i][j] = x[j + 1][i] - x[0][i];
  const double c00 = J[1][1] * J[2][2] - J[1][2] * J[2][1];
  const double c01 = J[1][2] * J[2][0] - J[1][0] * J[2][2];
  const double c02 = J[1][0] * J[2][1] - J[1][1] * J[2][0];
  const double det = J[0][0] * c00 + J[0][1] * c01 + J[0][2] * c02;
  const double idet = 1.0 / det;
  double g[4][3];
  g[1][0] = c00 * idet; g[2][0] = c01 * idet; g[3][0] = c02 * idet;
  g[1][1] = (J[0][2] * J[2][1] - J[0][1] * J[2][2]) * idet;
  g[2][1] = (J[0][0] * J[2][2] - J[0][2] * J[2][0]) * idet;
  g[3][1] = (J[0][1] * J[2][0] - J[0][0] * J[2][1]) * idet;
  g[1][2] = (J[0][1] * J[1][2] - J[0][2] * J[1][1]) * idet;
  g[2][2] = (J[0][2] * J[1][0] - J[0][0] * J[1][2]) * idet;
  g[3][2] = (J[0][0] * J[1][1] - J[0][1] * J[1][0]) * idet;
#pragma unroll
  for (int j = 0; j < 3; ++j) g[0][j] = -(g[1][j] + g[2][j] + g[3][j]);
  // the caller may pin a synchronisation point here (after the geometry, before anything is parked): it gets the weight and
  // hands it back, which ties every later quadrature sum to that point
  const double W = scratch.after_geometry(fabs(det) * (1.0 / 24.0));
  const double V = 4.0 * W;

  double G[6], gk[3];   // G: xx xy xz yy yz zz (sum over the three non-origin vertices)
#pragma unroll
  for (int j = 0; j < 3; ++j) gk[j] = row_is_origin ? g[1][j] : g[0][j];
  G[0] = gk[0] * gk[0] + g[2][0] * g[2][0] + g[3][0] * g[3][0];
  G[1] = gk[0] * gk[1] + g[2][0] * g[2][1] + g[3][0] * g[3][1];
  G[2] = gk[0] * gk[2] + g[2][0] * g[2][2] + g[3][0] * g[3][2];
  G[3] = gk[1] * gk[1] + g[2][1] * g[2][1] + g[3][1] * g[3][1];
  G[4] = gk[1] * gk[2] + g[2][1] * g[2][2] + g[3][1] * g[3][2];
  G[5] = gk[2] * gk[2] + g[2][2] * g[2][2] + g[3][2] * g[3][2];
  const double trG = G[0] + G[3] + G[5];
  const double Cst = fp.Ci * fp.nu * fp.nu * (G[0] * G[0] + G[3] * G[3] + G[5] * G[5] + 2.0 * (G[1] * G[1] + G[2] * G[2] + G[4] * G[4]));
  const double itrG = 1.0 / trG;

  double D[3][3], P[3], U[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    U[i] = u[0][i] + u[1][i] + u[2][i] + u[3][i];
#pragma unroll
    for (int j = 0; j < 3; ++j) D[i][j] = u[0][i] * g[0][j] + u[1][i] * g[1][j] + u[2][i] * g[2][j] + u[3][i] * g[3][j];
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) P[j] = p[0] * g[0][j] + p[1] * g[1][j] + p[2] * g[2][j] + p[3] * g[3][j];
  const double divu = D[0][0] + D[1][1] + D[2][2];

  // row-vertex constants needed inside the point loop: H = D g_0 and P . g_0, so that the SUPG weight a_0(q) = r_q . g_0
  // (r_q = grad p + u_q . grad u) is P.g_0 + H.u_q -- the residual vector r_q itself is never formed
  double H[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) H[d] = D[d][0] * g[0][0] + D[d][1] * g[0][1] + D[d][2] * g[0][2];
  const double Pg0 = P[0] * g[0][0] + P[1] * g[0][1] + P[2] * g[0][2];
  // the point loop needs neither grad u nor the gradients of the other three vertices: the caller may take them out of the
  // register file until the block loop (tensor-memory or shared-memory scratch in the kernels)
  scratch.put_geom(g, D);

  // ---- quadrature points: totals stay in registers, the data of points 1..3 is parked ----
  // (sum_q W tau r_q and sum_q W tau G u_q follow from s = sum_q W tau u_q after the loop: both are linear in u_q)
  double s[3] = {0, 0, 0}, Q[6] = {0, 0, 0, 0, 0, 0}, Y3[3] = {0, 0, 0}, sup[3] = {0, 0, 0};
  double Y1[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
  double tbar = 0.0, nuLbar = 0.0;
  P1TetPoint pt0;
  double ub[3];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    P1TetPoint pt;
#pragma unroll
    for (int i = 0; i < 3; ++i) pt.uq[i] = P1T_A * U[i] + P1T_E * u[q][i];
    pt.Gu[0] = G[0] * pt.uq[0] + G[1] * pt.uq[1] + G[2] * pt.uq[2];
    pt.Gu[1] = G[1] * pt.uq[0] + G[3] * pt.uq[1] + G[4] * pt.uq[2];
    pt.Gu[2] = G[2] * pt.uq[0] + G[4] * pt.uq[1] + G[5] * pt.uq[2];
    const double arg = Cst + pt.uq[0] * pt.Gu[0] + pt.uq[1] * pt.Gu[1] + pt.uq[2] * pt.Gu[2];
    const double tau = NS_RSQRT(arg);
    const double wt = W * tau;
    const double al = wt * (Pg0 + H[0] * pt.uq[0] + H[1] * pt.uq[1] + H[2] * pt.uq[2]);
    const double be = al * tau * tau;
    pt.ew = P1T_E * wt; pt.eb = P1T_E * be; pt.ea = P1T_E * al;
    tbar += wt;
    nuLbar += wt * arg;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      s[i] += wt * pt.uq[i];
      Y3[i] += be * pt.Gu[i];
      if (WANT_F) sup[i] += al * pt.uq[i];
    }
    {
      const double w0 = wt * pt.uq[0], w1 = wt * pt.uq[1], w2 = wt * pt.uq[2];
      Q[0] += w0 * pt.uq[0]; Q[1] += w0 * pt.uq[1]; Q[2] += w0 * pt.uq[2];
      Q[3] += w1 * pt.uq[1]; Q[4] += w1 * pt.uq[2]; Q[5] += w2 * pt.uq[2];
    }
    if (WANT_J) {
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const double bg = be * pt.Gu[d];
#pragma unroll
        for (int c = 0; c < 3; ++c) Y1[d][c] += bg * pt.uq[c];
      }
    }
    if (q == 0) {
      pt0 = pt;
#pragma unroll
      for (int d = 0; d < 3; ++d) ub[d] = W * (P1T_A * U[d] + P1T_E * pt.uq[d]);   // sum_q W N_0(q) u_q
    } else if (WANT_J) {
      scratch.put(q, pt);
    }
  }
  nuLbar *= itrG;

  const double TR0 = tbar * Pg0 + H[0] * s[0] + H[1] * s[1] + H[2] * s[2];   // (sum_q W tau r_q) . g_0
  scratch.get_D(D);

  if (WANT_F) {
    const double pbarV = W * (p[0] + p[1] + p[2] + p[3]);
#pragma unroll
    for (int c = 0; c < 3; ++c)
      fr[c] = D[c][0] * ub[0] + D[c][1] * ub[1] + D[c][2] * ub[2] + fp.nu * V * H[c] - pbarV * g[0][c] + sup[c] + nuLbar * divu * g[0][c];
    fr[3] = W * divu + TR0;
  }

  if (WANT_J) {
    const double kap = divu * itrG;
    const double M_off = W * (4.0 * P1T_A * P1T_A + 2.0 * P1T_A * P1T_E);
    const double akap = P1T_A * kap;
    // column-vertex independent parts
    const double ZG[3] = {G[0] * s[0] + G[1] * s[1] + G[2] * s[2], G[1] * s[0] + G[3] * s[1] + G[4] * s[2],
                          G[2] * s[0] + G[4] * s[1] + G[5] * s[2]};   // sum_q W tau G u_q = G s
    double C0[3][3], P0[3];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int d = 0; d < 3; ++d)
        C0[c][d] = M_off * D[c][d] + P1T_A * (s[c] * H[d] - Y1[d][c]) + akap * ZG[d] * g[0][c];
#pragma unroll
    for (int d = 0; d < 3; ++d) P0[d] = P1T_A * (tbar * H[d] - Y3[d]);
    const double dia0 = P1T_A * TR0;
    const double nuV = fp.nu * V;
    const double Qm[3][3] = {{Q[0], Q[1], Q[2]}, {Q[1], Q[3], Q[4]}, {Q[2], Q[4], Q[5]}};
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      P1TetPoint pt;
      if (n == 0) pt = pt0; else { scratch.get(n, pt); scratch.get_g(n, g[n]); }
      const double L = g[0][0] * g[n][0] + g[0][1] * g[n][1] + g[0][2] * g[n][2];
      double t1[3], t2[3];
      const double ewk = pt.ew * kap;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        t1[d] = pt.ew * H[d] - pt.eb * pt.Gu[d];
        t2[d] = ewk * pt.Gu[d] + nuLbar * g[n][d];
      }
      const double dia = ub[0] * g[n][0] + ub[1] * g[n][1] + ub[2] * g[n][2] + nuV * L + dia0 + pt.ea;
      double blk[16];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          double v = C0[c][d] + L * Qm[c][d] + pt.uq[c] * t1[d] + g[0][c] * t2[d];
          if (n == 0) v += (W * P1T_E * P1T_E) * D[c][d];
          if (c == d) v += dia;
          blk[4 * c + d] = v;
        }
        blk[4 * c + 3] = s[c] * L - W * g[0][c];
      }
#pragma unroll
      for (int d = 0; d < 3; ++d) blk[12 + d] = P0[d] + W * g[n][d] + t1[d] + s[d] * L;
      blk[15] = tbar * L;
      // a scratch kept outside the caller's output area lets the caller wait for that area only here; no lane-divergent branch
      // in this function encloses the block loop, so every thread of a warp that runs it reaches this point
      if (n == 0) scratch.before_first_emit();
      emit(n, blk);
    }
  }
}

}  // namespace nsgpu
struct nsgpu_ctx;
namespace nsgpu {
bool p1tet_fast_available(nsgpu_ctx* ctx);
int p1tet_assemble(nsgpu_ctx* ctx, const double* d_xin, bool want_J, bool want_F, double* d_Fout, int part = 0, int sm_reserve = 0);
bool p1tet_can_split(nsgpu_ctx* ctx);
int p1tet_build_plan(nsgpu_ctx* ctx);
void p1tet_free(nsgpu_ctx* ctx);
void p1tet_mark_bc_dirty(nsgpu_ctx* ctx);
int p1tet_spmv(nsgpu_ctx* ctx, const double* d_x, double* d_y);
// the vertex-blocked view of the CSR matrix the block SpMV walks (also used by the block ILU, ilu.cu): per vertex the start of its
// neighbour list in ctx->d_pairs, the number of neighbours, the CSR starts of its four rows and its four dofs
struct P1BlockView { int64_t n_ent; const int64_t* pair0; const int32_t* ns; const int64_t* rowpos; const int32_t* rowdof; };
bool p1tet_block_view(nsgpu_ctx* ctx, P1BlockView* out);
int p1tet_assemble_streamed(nsgpu_ctx* ctx, const double* x_host, double* F_host);
}  // namespace nsgpu
