// trace_core.cuh -- one streamline of a P1 velocity field on a tetrahedral mesh: point location, velocity
// evaluation and the adaptive Dormand-Prince integrator with terminal events, per seed, in one thread.
//
// Replaces the per-seed scipy.integrate.solve_ivp(velfunc, (0, 20), seed, method='RK45', events=..., max_step=0.125)
// calls of NavierStokes/streamtrace.py:198-218 (forward) and :357-384 (reverse), whose right-hand side
// velfunc (:144-158) locates the point with dolfinx's bounding-box tree + compute_colliding_cells and evaluates
// uh.eval; outside the mesh the velocity is zero.  The integrator follows scipy 1.x's RK45 step by step
// (select_initial_step, the error-norm step controller with SAFETY 0.9 / MIN_FACTOR 0.2 / MAX_FACTOR 10, the quartic
// dense output and root finding of terminal events on it) so that the end points agree with the reference's to
// rounding, not just to the integration tolerance.
//
// Everything here is __host__ __device__: tests compile the same code with g++ to compare it with scipy on the CPU.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define TR_HD __host__ __device__ __forceinline__
#else
#define TR_HD inline
#endif

namespace nsgpu {

// Locator + field tables (device pointers in the library, host pointers in the test harness); the locator part is a view of
// the context's Locator (csrc/locate.cu)
struct TraceField {
  const double* cmap;      // per cell 12 doubles: x0[3], K[3][3] (row a = gradient of barycentric coordinate a+1)
  const double* cvel;      // per cell 12 doubles: c[3], A[3][3]  with  u(x) = c + A x
  const int64_t* bin_ptr;  // nbx*nby*nbz + 1
  const int32_t* bin_cells;
  double lo[3], inv_h[3];
  int nb[3];
  double tol;              // a point is inside a cell when every barycentric coordinate is >= -tol
};

struct TraceParams {
  double dir;        // +1: trace along u (streamtrace.py:144), -1: along -u (velfunc_reverese, :160)
  double x_stop;     // position event  y[0] - x_stop  (:183 forward 3.7, :188 reverse 0.13)
  double x_dir;      // its direction (+1 forward :207, -1 reverse :362)
  double speed_min;  // velocity event  |u| - speed_min, direction -1 (:177-180, 1e-6)
  double t_end, max_step, rtol, atol;
  int64_t max_steps;
};

enum { TRACE_FINISHED = 0, TRACE_EVENT_POSITION = 1, TRACE_EVENT_SPEED = 2, TRACE_STEP_TOO_SMALL = -1, TRACE_MAX_STEPS = -2 };

// ---- point locator queries (the tables are built by csrc/locate.cu; also used by the point evaluation there) ----
// cmap row of a cell: x0[GD], then K[GD][GD] with row a = gradient of barycentric coordinate a+1
template <int GD> TR_HD void loc_bary(const double* cmap, int32_t c, const double* p, double* l) {
  if constexpr (GD == 3) {
    const double* m = cmap + 12 * (int64_t)c;
    const double d0 = p[0] - m[0], d1 = p[1] - m[1], d2 = p[2] - m[2];
    l[1] = m[3] * d0 + m[4] * d1 + m[5] * d2;
    l[2] = m[6] * d0 + m[7] * d1 + m[8] * d2;
    l[3] = m[9] * d0 + m[10] * d1 + m[11] * d2;
    l[0] = 1.0 - l[1] - l[2] - l[3];
  } else {
    const double* m = cmap + 6 * (int64_t)c;
    const double d0 = p[0] - m[0], d1 = p[1] - m[1];
    l[1] = m[2] * d0 + m[3] * d1;
    l[2] = m[4] * d0 + m[5] * d1;
    l[0] = 1.0 - l[1] - l[2];
  }
}

// inside = every barycentric coordinate >= -tol
template <int GD> TR_HD bool loc_inside(const double* cmap, int32_t c, const double* p, double tol) {
  double l[GD + 1];
  loc_bary<GD>(cmap, c, p, l);
  const double t = -tol;
  bool in = true;
  for (int a = 0; a <= GD; ++a) in = in && l[a] >= t;
  return in;
}

// lowest-numbered cell below n_bound of p's bin that holds p; -1 when none does (or p is off the grid).  The grid has one layer in z
// for GD = 2.  The bin lists are ascending, so the scan stops at the first cell >= n_bound (several ranks: the owned cells only).
template <int GD> TR_HD int32_t loc_find(const double* cmap, const int64_t* bin_ptr, const int32_t* bin_cells, const double* lo,
                                         const double* inv_h, const int* nb, int32_t n_bound, double tol, const double* p) {
  int b[3] = {0, 0, 0};
  for (int k = 0; k < GD; ++k) {
    const double s = (p[k] - lo[k]) * inv_h[k];
    if (!(s >= 0.0) || s >= (double)nb[k] + 1e-9) return -1;
    int i = (int)s;
    b[k] = i >= nb[k] ? nb[k] - 1 : i;
  }
  const int64_t bin = ((int64_t)b[2] * nb[1] + b[1]) * nb[0] + b[0];
  for (int64_t k = bin_ptr[bin]; k < bin_ptr[bin + 1]; ++k) {
    const int32_t c = bin_cells[k];
    if (c >= n_bound) break;
    if (loc_inside<GD>(cmap, c, p, tol)) return c;
  }
  return -1;
}

TR_HD bool tr_inside(const TraceField& F, int32_t c, const double* p) { return loc_inside<3>(F.cmap, c, p, F.tol); }

// cell holding p: the cached cell if it still does, else the lowest-numbered cell of p's bin that does; -1 outside the mesh
TR_HD int32_t tr_locate(const TraceField& F, const double* p, int32_t hint) {
  if (hint >= 0 && tr_inside(F, hint, p)) return hint;
  return loc_find<3>(F.cmap, F.bin_ptr, F.bin_cells, F.lo, F.inv_h, F.nb, INT32_MAX, F.tol, p);   // every cell of the mesh
}

// velfunc / velfunc_reverese: dir * u(p), zero outside the mesh
TR_HD void tr_velocity(const TraceField& F, double dir, const double* p, int32_t& cell, double* v) {
  cell = tr_locate(F, p, cell);
  if (cell < 0) { v[0] = v[1] = v[2] = 0.0; return; }
  const double* a = F.cvel + 12 * (int64_t)cell;
  for (int i = 0; i < 3; ++i) v[i] = dir * (a[i] + a[3 + 3 * i] * p[0] + a[4 + 3 * i] * p[1] + a[5 + 3 * i] * p[2]);
}

TR_HD double tr_rms3(double a, double b, double c) { return sqrt((a * a + b * b + c * c) / 3.0); }

// dense output of the accepted step (scipy RkDenseOutput): y(t) = y_old + h * Q p,  p = (x, x^2, x^3, x^4)
struct TraceDense {
  double t_old, h, y_old[3], Q[3][4];
  TR_HD void eval(double t, double* y) const {
    const double x = (t - t_old) / h;
    const double x2 = x * x, x3 = x2 * x, x4 = x3 * x;
    for (int i = 0; i < 3; ++i) y[i] = h * (Q[i][0] * x + Q[i][1] * x2 + Q[i][2] * x3 + Q[i][3] * x4) + y_old[i];
  }
};

// event functions on the dense output (streamtrace.py:177-190)
TR_HD double tr_event(const TraceField& F, const TraceParams& P, const TraceDense& D, int which, double t, int32_t& cell) {
  double y[3];
  D.eval(t, y);
  if (which == 0) return y[0] - P.x_stop;
  double v[3];
  tr_velocity(F, 1.0, y, cell, v);
  return sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]) - P.speed_min;
}

// Brent's bracketing root finder with scipy.optimize.brentq's tolerances (xtol = rtol = 4 eps): root of event(t) in [a, b]
TR_HD double tr_brent(const TraceField& F, const TraceParams& P, const TraceDense& D, int which, double xa, double xb, int32_t& cell) {
  const double xtol = 4.0 * 2.220446049250313e-16, rtol = 4.0 * 2.220446049250313e-16;
  double xpre = xa, xcur = xb, xblk = 0.0, fblk = 0.0, spre = 0.0, scur = 0.0;
  double fpre = tr_event(F, P, D, which, xpre, cell);
  double fcur = tr_event(F, P, D, which, xcur, cell);
  if (fpre == 0.0) return xpre;
  if (fcur == 0.0) return xcur;
  for (int it = 0; it < 100; ++it) {
    if (fpre != 0.0 && fcur != 0.0 && ((fpre < 0.0) != (fcur < 0.0))) { xblk = xpre; fblk = fpre; spre = scur = xcur - xpre; }
    if (fabs(fblk) < fabs(fcur)) { xpre = xcur; xcur = xblk; xblk = xpre; fpre = fcur; fcur = fblk; fblk = fpre; }
    const double delta = (xtol + rtol * fabs(xcur)) / 2.0;
    const double sbis = (xblk - xcur) / 2.0;
    if (fcur == 0.0 || fabs(sbis) < delta) return xcur;
    if (fabs(spre) > delta && fabs(fcur) < fabs(fpre)) {
      double stry;
      if (xpre == xblk) stry = -fcur * (xcur - xpre) / (fcur - fpre);   // secant
      else {                                                            // inverse quadratic extrapolation
        const double dpre = (fpre - fcur) / (xpre - xcur), dblk = (fblk - fcur) / (xblk - xcur);
        stry = -fcur * (fblk * dblk - fpre * dpre) / (dblk * dpre * (fblk - fpre));
      }
      const double lim1 = fabs(spre), lim2 = 3.0 * fabs(sbis) - delta;
      if (2.0 * fabs(stry) < (lim1 < lim2 ? lim1 : lim2)) { spre = scur; scur = stry; }
      else { spre = sbis; scur = sbis; }
    } else { spre = sbis; scur = sbis; }
    xpre = xcur; fpre = fcur;
    if (fabs(scur) > delta) xcur += scur;
    else xcur += (sbis > 0.0 ? delta : -delta);
    fcur = tr_event(F, P, D, which, xcur, cell);
  }
  return xcur;
}

struct TraceResult {
  double y[3], t;
  int32_t status, n_steps, n_fev;
};

// One seed, start to finish (= one solve_ivp call of streamtrace_pool / reverse_streamtrace_pool).
TR_HD void tr_trace(const TraceField& F, const TraceParams& P, const double* seed, TraceResult& R) {
  // Dormand-Prince 5(4) tableau (scipy.integrate._ivp.rk.RK45)
  const double C1 = 1.0 / 5, C2 = 3.0 / 10, C3 = 4.0 / 5, C4 = 8.0 / 9;
  const double A10 = 1.0 / 5;
  const double A20 = 3.0 / 40, A21 = 9.0 / 40;
  const double A30 = 44.0 / 45, A31 = -56.0 / 15, A32 = 32.0 / 9;
  const double A40 = 19372.0 / 6561, A41 = -25360.0 / 2187, A42 = 64448.0 / 6561, A43 = -212.0 / 729;
  const double A50 = 9017.0 / 3168, A51 = -355.0 / 33, A52 = 46732.0 / 5247, A53 = 49.0 / 176, A54 = -5103.0 / 18656;
  const double B0 = 35.0 / 384, B2 = 500.0 / 1113, B3 = 125.0 / 192, B4 = -2187.0 / 6784, B5 = 11.0 / 84;
  const double E0 = -71.0 / 57600, E2 = 71.0 / 16695, E3 = -71.0 / 1920, E4 = 17253.0 / 339200, E5 = -22.0 / 525, E6 = 1.0 / 40;
  const double PM[7][4] = {
      {1.0, -8048581381.0 / 2820520608.0, 8663915743.0 / 2820520608.0, -12715105075.0 / 11282082432.0},
      {0.0, 0.0, 0.0, 0.0},
      {0.0, 131558114200.0 / 32700410799.0, -68118460800.0 / 10900136933.0, 87487479700.0 / 32700410799.0},
      {0.0, -1754552775.0 / 470086768.0, 14199869525.0 / 1410260304.0, -10690763975.0 / 1880347072.0},
      {0.0, 127303824393.0 / 49829197408.0, -318862633887.0 / 49829197408.0, 701980252875.0 / 199316789632.0},
      {0.0, -282668133.0 / 205662961.0, 2019193451.0 / 616988883.0, -1453857185.0 / 822651844.0},
      {0.0, 40617522.0 / 29380423.0, -110615467.0 / 29380423.0, 69997945.0 / 29380423.0}};
  const double SAFETY = 0.9, MIN_FACTOR = 0.2, MAX_FACTOR = 10.0, EXPO = -1.0 / 5.0;

  double t = 0.0, y[3] = {seed[0], seed[1], seed[2]}, f[3];
  int32_t cell = -1;
  int32_t n_fev = 0, n_steps = 0;
  tr_velocity(F, P.dir, y, cell, f); ++n_fev;

  // select_initial_step (order 4 error estimator)
  double h_abs;
  {
    const double interval = fabs(P.t_end - t);
    double sc[3];
    for (int i = 0; i < 3; ++i) sc[i] = P.atol + fabs(y[i]) * P.rtol;
    const double d0 = tr_rms3(y[0] / sc[0], y[1] / sc[1], y[2] / sc[2]);
    const double d1 = tr_rms3(f[0] / sc[0], f[1] / sc[1], f[2] / sc[2]);
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
    h0 = h0 < interval ? h0 : interval;
    double y1[3], f1[3];
    for (int i = 0; i < 3; ++i) y1[i] = y[i] + h0 * f[i];
    int32_t c1 = cell;
    tr_velocity(F, P.dir, y1, c1, f1); ++n_fev;
    const double d2 = tr_rms3((f1[0] - f[0]) / sc[0], (f1[1] - f[1]) / sc[1], (f1[2] - f[2]) / sc[2]) / h0;
    double h1;
    if (d1 <= 1e-15 && d2 <= 1e-15) h1 = (1e-6 > h0 * 1e-3) ? 1e-6 : h0 * 1e-3;
    else h1 = pow(0.01 / (d1 > d2 ? d1 : d2), 1.0 / 5.0);
    h_abs = 100.0 * h0;
    if (h1 < h_abs) h_abs = h1;
    if (interval < h_abs) h_abs = interval;
    if (P.max_step < h_abs) h_abs = P.max_step;
  }

  // event values at the start (solve_ivp: g = [event(t0, y0) ...])
  double g_pos = y[0] - P.x_stop;
  double g_spd = sqrt(f[0] * f[0] + f[1] * f[1] + f[2] * f[2]) - P.speed_min;

  int32_t status = TRACE_FINISHED;
  while (true) {
    if (t == P.t_end) { status = TRACE_FINISHED; break; }
    if (n_steps >= P.max_steps) { status = TRACE_MAX_STEPS; break; }
    const double min_step = 10.0 * fabs(nextafter(t, INFINITY) - t);
    if (h_abs > P.max_step) h_abs = P.max_step;
    else if (h_abs < min_step) h_abs = min_step;

    double K[7][3], y_new[3], f_new[3], h = 0.0, t_new = t;
    bool rejected = false, failed = false;
    int32_t c_new = cell;
    while (true) {
      if (h_abs < min_step) { failed = true; break; }
      h = h_abs;
      t_new = t + h;
      if (t_new - P.t_end > 0.0) t_new = P.t_end;
      h = t_new - t;
      h_abs = fabs(h);
      // rk_step
      double ys[3];
      int32_t cs = cell;
      for (int i = 0; i < 3; ++i) { K[0][i] = f[i]; ys[i] = y[i] + (K[0][i] * A10) * h; }
      tr_velocity(F, P.dir, ys, cs, K[1]);
      for (int i = 0; i < 3; ++i) ys[i] = y[i] + (K[0][i] * A20 + K[1][i] * A21) * h;
      tr_velocity(F, P.dir, ys, cs, K[2]);
      for (int i = 0; i < 3; ++i) ys[i] = y[i] + (K[0][i] * A30 + K[1][i] * A31 + K[2][i] * A32) * h;
      tr_velocity(F, P.dir, ys, cs, K[3]);
      for (int i = 0; i < 3; ++i) ys[i] = y[i] + (K[0][i] * A40 + K[1][i] * A41 + K[2][i] * A42 + K[3][i] * A43) * h;
      tr_velocity(F, P.dir, ys, cs, K[4]);
      for (int i = 0; i < 3; ++i) ys[i] = y[i] + (K[0][i] * A50 + K[1][i] * A51 + K[2][i] * A52 + K[3][i] * A53 + K[4][i] * A54) * h;
      tr_velocity(F, P.dir, ys, cs, K[5]);
      for (int i = 0; i < 3; ++i) y_new[i] = y[i] + h * (K[0][i] * B0 + K[2][i] * B2 + K[3][i] * B3 + K[4][i] * B4 + K[5][i] * B5);
      tr_velocity(F, P.dir, y_new, cs, f_new);
      n_fev += 6;
      (void)C1; (void)C2; (void)C3; (void)C4;   // the field is autonomous: stage times are not needed
      for (int i = 0; i < 3; ++i) K[6][i] = f_new[i];
      double en2 = 0.0;
      for (int i = 0; i < 3; ++i) {
        const double ay = fabs(y[i]), an = fabs(y_new[i]);
        const double scale = P.atol + (ay > an ? ay : an) * P.rtol;
        const double e = (K[0][i] * E0 + K[2][i] * E2 + K[3][i] * E3 + K[4][i] * E4 + K[5][i] * E5 + K[6][i] * E6) * h / scale;
        en2 += e * e;
      }
      const double err = sqrt(en2 / 3.0);
      if (err < 1.0) {
        double factor = (err == 0.0) ? MAX_FACTOR : SAFETY * pow(err, EXPO);
        if (factor > MAX_FACTOR) factor = MAX_FACTOR;
        if (rejected && factor > 1.0) factor = 1.0;
        h_abs *= factor;
        c_new = cs;
        break;
      }
      const double fac = SAFETY * pow(err, EXPO);
      h_abs *= (fac > MIN_FACTOR ? fac : MIN_FACTOR);
      rejected = true;
    }
    if (failed) { status = TRACE_STEP_TOO_SMALL; break; }
    ++n_steps;

    // events on the accepted step (find_active_events / handle_events / solve_event_equation)
    const double gn_pos = y_new[0] - P.x_stop;
    const double gn_spd = sqrt(f_new[0] * f_new[0] + f_new[1] * f_new[1] + f_new[2] * f_new[2]) - P.speed_min;
    const bool up_pos = g_pos <= 0.0 && gn_pos >= 0.0, down_pos = g_pos >= 0.0 && gn_pos <= 0.0;
    const bool act_pos = P.x_dir > 0.0 ? up_pos : down_pos;
    const bool act_spd = g_spd >= 0.0 && gn_spd <= 0.0;   // direction -1
    if (act_pos || act_spd) {
      TraceDense D;
      D.t_old = t; D.h = h;
      for (int i = 0; i < 3; ++i) {
        D.y_old[i] = y[i];
        for (int j = 0; j < 4; ++j) {
          double s = 0.0;
          for (int k = 0; k < 7; ++k) s += K[k][i] * PM[k][j];
          D.Q[i][j] = s;
        }
      }
      int32_t ce = c_new;
      double te = 0.0;
      int which = -1;
      if (act_pos) { te = tr_brent(F, P, D, 0, t, t_new, ce); which = 0; }
      if (act_spd) {
        const double ts = tr_brent(F, P, D, 1, t, t_new, ce);
        if (which < 0 || ts < te) { te = ts; which = 1; }
      }
      D.eval(te, y);
      t = te;
      status = which == 0 ? TRACE_EVENT_POSITION : TRACE_EVENT_SPEED;
      break;
    }
    g_pos = gn_pos; g_spd = gn_spd;
    t = t_new;
    for (int i = 0; i < 3; ++i) { y[i] = y_new[i]; f[i] = f_new[i]; }
    cell = c_new;
  }
  R.y[0] = y[0]; R.y[1] = y[1]; R.y[2] = y[2];
  R.t = t; R.status = status; R.n_steps = n_steps; R.n_fev = n_fev;
}

}  // namespace nsgpu
