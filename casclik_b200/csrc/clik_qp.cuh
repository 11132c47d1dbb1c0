// clik_qp.cuh — batched dense strictly-convex QP for the reactive-QP controller step, one
// instance per thread, fp64, sm_100a.
//
//     min 1/2 x' diag(h) x      s.t.  lb <= A x <= ub            x = [robot vel; virtual vel; slack]
//
// This is the problem the reference assembles in ReactiveQPController.get_cost_expr /
// get_constraints_expr (reference casclik/controllers/reactive_qp.py:175-246) and hands to
// qpOASES through cs.conic (:256-260, :493, :512-513).  h > 0 (mu*w, mu + w_slack), so the
// minimiser is unique and any exact method returns the point qpOASES converges to.
//
// Method: Goldfarb-Idnani dual active set in the coordinates z = sqrt(h) .* x, where the
// objective is 1/2 |z|^2 and there is no linear term (the reference never passes g).  z starts at
// the unconstrained minimiser 0; each outer iteration picks the most violated one-sided
// constraint and walks to it along the projection of its normal onto the null space of the active
// normals, dropping active constraints whose multiplier would turn negative.  The active normals
// are re-orthogonalised from scratch (modified Gram-Schmidt, at most NX columns) whenever the
// working set changes: the matrices are tiny (UR5 config: 9 x 15) and it keeps the projection
// accurate without squaring the condition number.  The iteration count is capped (status 1).
// (This is the generic dense variant; skills with few dense rows use qp_structured below, which
// also accepts warm starts.)
//
// Outputs per instance: x, status (0 solved, 1 iteration cap, 2 infeasible), and two bit masks
// of the rows active at their upper / lower bound in the final working set.
#pragma once
#include <cstdint>
#include <cmath>

namespace clik {

enum : int { QP_OK = 0, QP_MAXITER = 1, QP_INFEASIBLE = 2, QP_PENDING = 3 /* transient: between the fast and the tail pass */,
             QP_INVALID = 4 /* non-finite problem data or solution (NaN inputs, non-positive cost weight) */ };

// A solution containing NaN / inf is never reported as solved (a zero cost weight makes 1/sqrt(h) infinite,
// a NaN input poisons every comparison of the iteration, which then "finds no violated row").
// inf / NaN test on the high word (integer pipe): exponent field all ones
__device__ __forceinline__ bool finite_bits(double v) {
  return (__double2hiint(v) & 0x7ff00000) != 0x7ff00000;
}
__device__ __forceinline__ constexpr bool row_read(unsigned mask, int j) { return j >= 32 || ((mask >> j) & 1u) != 0u; }
template <int N> __device__ __forceinline__ bool all_finite(const double (&x)[N]) {
  bool ok = true;
#pragma unroll
  for (int j = 0; j < N; ++j) ok = ok && (fabs(x[j]) < INFINITY);
  return ok;
}

// NXM / MM: compile-time capacities; nx / m: actual sizes (compile-time constants when inlined
// into a fused skill kernel).  A is row-major m x nx and is overwritten with the scaled rows.
template <int NXM, int MM>
__device__ int qp_dual_active_set(const int nx, const int m, double* A, const double* lb,
                                  const double* ub, const double* h, const double* x0, double* x,
                                  unsigned* act_up, unsigned* act_lo, const int max_iter) {
  double s[NXM], z[NXM], d[NXM], np_[NXM], c[NXM], rr[NXM], u[NXM];
  double Qb[NXM * NXM];   // orthonormal basis of the active normals, column a at Qb[a*nx .. )
  double R[NXM * NXM];    // upper triangular, R[l*NXM + a]
  int W[NXM];
  signed char state[MM];
  int k = 0;

  for (int j = 0; j < nx; ++j) {
    s[j] = rsqrt(h[j]);
    z[j] = 0.0;
  }
  for (int i = 0; i < m; ++i) {
    state[i] = 0;
    for (int j = 0; j < nx; ++j) A[i * nx + j] *= s[j];
  }
  (void)x0;  // primal warm start: the dual method restarts from z = 0 (result is independent of x0)

  int status = QP_MAXITER;
  bool need_qr = false;
  for (int it = 0; it < max_iter; ++it) {
    // ---- most violated one-sided constraint ------------------------------------------------
    int p = -1;
    double sp = 0.0, vbest = 0.0;
    for (int i = 0; i < m; ++i) {
      if (state[i] != 0) continue;
      double r = 0.0;
      for (int j = 0; j < nx; ++j) r = fma(A[i * nx + j], z[j], r);
      const double vu = r - ub[i], vl = lb[i] - r;
      const double tu = 1e-12 * fmax(1.0, fabs(ub[i])), tl = 1e-12 * fmax(1.0, fabs(lb[i]));
      if (vu > tu && vu > vbest) { vbest = vu; p = i; sp = 1.0; }
      if (vl > tl && vl > vbest) { vbest = vl; p = i; sp = -1.0; }
    }
    if (p < 0) { status = QP_OK; break; }

    double nn = 0.0;
    for (int j = 0; j < nx; ++j) { np_[j] = sp * A[p * nx + j]; nn = fma(np_[j], np_[j], nn); }
    double up = 0.0;
    bool done = false, infeasible = false;
    while (!done) {
      // ---- (re)factor the active normals: N = Qb R ----------------------------------------
      if (need_qr) {
        for (int a = 0; a < k; ++a) {
          const double sg = (double)state[W[a]];
          double* col = &Qb[a * nx];
          for (int j = 0; j < nx; ++j) col[j] = sg * A[W[a] * nx + j];
          for (int pass = 0; pass < 2; ++pass) {
            for (int l = 0; l < a; ++l) {
              double dt = 0.0;
              for (int j = 0; j < nx; ++j) dt = fma(Qb[l * nx + j], col[j], dt);
              for (int j = 0; j < nx; ++j) col[j] = fma(-dt, Qb[l * nx + j], col[j]);
              R[l * NXM + a] = (pass == 0) ? dt : R[l * NXM + a] + dt;
            }
          }
          double nrm = 0.0;
          for (int j = 0; j < nx; ++j) nrm = fma(col[j], col[j], nrm);
          nrm = sqrt(nrm);
          R[a * NXM + a] = nrm;
          const double inv = 1.0 / nrm;
          for (int j = 0; j < nx; ++j) col[j] *= inv;
        }
        need_qr = false;
      }
      // ---- d = (I - Qb Qb') n_p ,  r = R^-1 Qb' n_p ------------------------------------------
      for (int j = 0; j < nx; ++j) d[j] = np_[j];
      for (int a = 0; a < k; ++a) c[a] = 0.0;
      for (int pass = 0; pass < 2; ++pass) {
        for (int a = 0; a < k; ++a) {
          double dt = 0.0;
          for (int j = 0; j < nx; ++j) dt = fma(Qb[a * nx + j], d[j], dt);
          for (int j = 0; j < nx; ++j) d[j] = fma(-dt, Qb[a * nx + j], d[j]);
          c[a] += dt;
        }
      }
      for (int a = k - 1; a >= 0; --a) {
        double acc = c[a];
        for (int l = a + 1; l < k; ++l) acc = fma(-R[a * NXM + l], rr[l], acc);
        rr[a] = acc / R[a * NXM + a];
      }
      double dn = 0.0;
      for (int j = 0; j < nx; ++j) dn = fma(d[j], d[j], dn);
      // ---- step lengths -----------------------------------------------------------------------
      double rmax = 0.0;
      for (int a = 0; a < k; ++a) rmax = fmax(rmax, fabs(rr[a]));
      double t1 = INFINITY;
      int drop = -1;
      for (int a = 0; a < k; ++a) {
        if (rr[a] > 1e-12 * rmax && rr[a] > 0.0) {
          const double cand = u[a] / rr[a];
          if (cand < t1) { t1 = cand; drop = a; }
        }
      }
      double rp = 0.0;
      for (int j = 0; j < nx; ++j) rp = fma(A[p * nx + j], z[j], rp);
      const double viol = (sp > 0.0) ? (rp - ub[p]) : (lb[p] - rp);
      const bool independent = (k < nx) && (dn > 1e-24 * nn);
      const double t2 = independent ? viol / dn : INFINITY;
      const double t = fmin(t1, t2);
      if (!(t < INFINITY)) { infeasible = true; break; }
      if (independent) {
        for (int j = 0; j < nx; ++j) z[j] = fma(-t, d[j], z[j]);
      }
      for (int a = 0; a < k; ++a) u[a] = fma(-t, rr[a], u[a]);
      up += t;
      if (t2 <= t1) {
        // full step: p joins the working set; extend the factorisation by one column
        W[k] = p;
        state[p] = (sp > 0.0) ? 1 : -1;
        u[k] = up;
        for (int a = 0; a < k; ++a) R[a * NXM + k] = c[a];
        const double nrm = sqrt(dn);
        R[k * NXM + k] = nrm;
        const double inv = 1.0 / nrm;
        for (int j = 0; j < nx; ++j) Qb[k * nx + j] = d[j] * inv;
        ++k;
        done = true;
      } else {
        // partial step: drop the blocking constraint and try again with the same p
        state[W[drop]] = 0;
        for (int a = drop; a < k - 1; ++a) { W[a] = W[a + 1]; u[a] = u[a + 1]; }
        --k;
        need_qr = true;
      }
    }
    if (infeasible) { status = QP_INFEASIBLE; break; }
  }

  for (int j = 0; j < nx; ++j) x[j] = z[j] * s[j];
  unsigned mu = 0u, ml = 0u;
  for (int a = 0; a < k; ++a) {
    if (W[a] < 32) {
      if (state[W[a]] > 0) mu |= 1u << W[a]; else ml |= 1u << W[a];
    }
  }
  *act_up = mu;
  *act_lo = ml;
  return status;
}

// ---- structured variant ---------------------------------------------------------------------------
// Most rows of a reactive-QP are bounds on single variables (joint-position limits and joint-speed
// limits are identity rows: reference reactive_qp.py:221-231 with expression = q), only the task
// rows are dense.  The expression compiler classifies the rows at compile time (S::QMD dense rows,
// S::QMU unit rows with constant coefficient S::unit_coef(i) on column S::unit_col(i)); this solver
// runs the same Goldfarb-Idnani iteration as qp_dual_active_set but keeps the working set as
//   * a set of fixed coordinates (active unit rows: their normals are coordinate vectors, so
//     projecting them out is just "zero that coordinate"), and
//   * a QR factorisation of the active dense normals restricted to the free coordinates,
// which is at most QMD columns.  Everything is indexed at compile time and lives in registers.
template <class S> struct QpSData {
  double Ad[(S::QMD > 0 ? S::QMD : 1) * S::QN];   // dense rows (unscaled on entry)
  double lbd[S::QMD > 0 ? S::QMD : 1], ubd[S::QMD > 0 ? S::QMD : 1];
  double lbu[S::QMU > 0 ? S::QMU : 1], ubu[S::QMU > 0 ? S::QMU : 1];
  double s[S::QN];                                 // 1 / sqrt(h_j)
};

// warm_up / warm_lo (optional, 0 = cold start): a guess of the final working set in the output
// format (bit r = original row r held at its upper / lower bound), e.g. the previous step's masks
// in a closed-loop rollout.  The guess is turned into a valid dual-feasible starting point (minimum-
// norm point on the guessed face, constraints with negative multipliers released, equality rows
// flipped to the side with a positive multiplier); the iteration then proceeds as usual, so the
// result does not depend on the guess.
template <class S>
__device__ __forceinline__ int qp_structured(QpSData<S>& D, double (&x)[S::QN], unsigned* act_up,
                                             unsigned* act_lo, const int max_iter,
                                             const unsigned warm_up = 0u, const unsigned warm_lo = 0u) {
  constexpr int NX = S::QN, MD = S::QMD, MU = S::QMU;
  constexpr int MD1 = MD > 0 ? MD : 1, MU1 = MU > 0 ? MU : 1;
  double z[NX], nF[NX], inF[NX], uF[NX];   // nF[j] != 0: coordinate j is fixed (entry of its normal; inF = 1/nF)
  int frow[NX], fside[NX];           // active unit row on coordinate j and the side it is held at
  double Qd[MD1 * NX], Rd[MD1 * MD1], iRd[MD1], uD[MD1], ks[MU1];   // iRd = 1 / diagonal of Rd
  int ad[MD1];                       // 0 inactive, +1 held at upper, -1 held at lower
  int nact = 0;
#pragma unroll
  for (int j = 0; j < NX; ++j) { z[j] = 0.0; nF[j] = 0.0; inF[j] = 0.0; uF[j] = 0.0; frow[j] = -1; fside[j] = 0; }
#pragma unroll
  for (int a = 0; a < MD; ++a) {
    ad[a] = 0; uD[a] = 0.0; iRd[a] = 0.0;
#pragma unroll
    for (int j = 0; j < NX; ++j) D.Ad[a * NX + j] *= D.s[j];
  }
#pragma unroll
  for (int i = 0; i < MU; ++i) ks[i] = S::unit_coef(i) * D.s[S::unit_col(i)];

  // QR of the active dense normals on the free coordinates, rebuilt in slot order.  Branch-free:
  // an inactive slot has a zero column (Qd row = 0, iRd = 0, its Rd entries = 0), so every loop
  // of the iteration can run over all MD slots without per-thread control flow.
  auto refactor = [&]() {
#pragma unroll
    for (int a = 0; a < MD; ++a) {
      const double sa = (double)ad[a];
      double col[NX];
#pragma unroll
      for (int j = 0; j < NX; ++j) col[j] = (nF[j] != 0.0) ? 0.0 : sa * D.Ad[a * NX + j];
#pragma unroll
      for (int l = 0; l < a; ++l) Rd[l * MD1 + a] = 0.0;
#pragma unroll
      for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
        for (int l = 0; l < a; ++l) {
          double dt = 0.0;
#pragma unroll
          for (int j = 0; j < NX; ++j) dt = fma(Qd[l * NX + j], col[j], dt);
#pragma unroll
          for (int j = 0; j < NX; ++j) col[j] = fma(-dt, Qd[l * NX + j], col[j]);
          Rd[l * MD1 + a] += dt;
        }
      }
      double nrm = 0.0;
#pragma unroll
      for (int j = 0; j < NX; ++j) nrm = fma(col[j], col[j], nrm);
      nrm = sqrt(nrm);
      Rd[a * MD1 + a] = nrm;
      const double inv = (ad[a] != 0) ? 1.0 / nrm : 0.0;
      iRd[a] = inv;
#pragma unroll
      for (int j = 0; j < NX; ++j) Qd[a * NX + j] = (ad[a] != 0) ? col[j] * inv : 0.0;
    }
  };
#pragma unroll
  for (int a = 0; a < MD; ++a) {
#pragma unroll
    for (int j = 0; j < NX; ++j) Qd[a * NX + j] = 0.0;
#pragma unroll
    for (int l = 0; l < MD; ++l) Rd[a * MD1 + l] = 0.0;
  }

  if ((warm_up | warm_lo) != 0u) {
    // ---- adopt the guessed working set ---------------------------------------------------------
#pragma unroll
    for (int i = 0; i < MU; ++i) {
      const bool up_ = S::unit_row(i) < 32 && ((warm_up >> S::unit_row(i)) & 1u);
      const bool lo_ = S::unit_row(i) < 32 && ((warm_lo >> S::unit_row(i)) & 1u);
      const double bnd = up_ ? D.ubu[i] : D.lbu[i];
      if ((up_ || lo_) && frow[S::unit_col(i)] < 0 && nact < NX && (fabs(bnd) < INFINITY)) {
        const double sgn = up_ ? 1.0 : -1.0;
        nF[S::unit_col(i)] = sgn * ks[i];
        inF[S::unit_col(i)] = 1.0 / (sgn * ks[i]);
        frow[S::unit_col(i)] = i;
        fside[S::unit_col(i)] = up_ ? 1 : -1;
        z[S::unit_col(i)] = bnd / ks[i];
        ++nact;
      }
    }
#pragma unroll
    for (int a = 0; a < MD; ++a) {
      const bool up_ = S::dense_row(a) < 32 && ((warm_up >> S::dense_row(a)) & 1u);
      const bool lo_ = S::dense_row(a) < 32 && ((warm_lo >> S::dense_row(a)) & 1u);
      const double bnd = up_ ? D.ubd[a] : D.lbd[a];
      if ((up_ || lo_) && nact < NX && (fabs(bnd) < INFINITY)) { ad[a] = up_ ? 1 : -1; ++nact; }
    }
    // release / flip until every multiplier is non-negative
    bool warm_ok = false;
    for (int round = 0; round <= 2 * NX + MD; ++round) {
      refactor();
      // a dense row that became dependent on the rest of the guess is dropped
      bool dropped = false;
#pragma unroll
      for (int a = 0; a < MD; ++a) {
        if (ad[a] != 0 && !(Rd[a * MD1 + a] > 1e-12)) { ad[a] = 0; --nact; dropped = true; }
      }
      if (dropped) continue;
      // minimum-norm point on the face: fixed coordinates at their bounds, free part = Qd Rd^-T rhs
      double y[MD1], ud[MD1];
#pragma unroll
      for (int a = 0; a < MD; ++a) {
        double rhs = (ad[a] > 0) ? D.ubd[a] : -D.lbd[a];
#pragma unroll
        for (int j = 0; j < NX; ++j) {
          if (nF[j] != 0.0) rhs = fma(-(double)ad[a] * D.Ad[a * NX + j], z[j], rhs);
        }
#pragma unroll
        for (int l = 0; l < a; ++l) {
          if (ad[l] != 0) rhs = fma(-Rd[l * MD1 + a], y[l], rhs);
        }
        y[a] = (ad[a] != 0) ? rhs * iRd[a] : 0.0;
      }
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        if (nF[j] == 0.0) {
          double acc = 0.0;
#pragma unroll
          for (int a = 0; a < MD; ++a) {
            if (ad[a] != 0) acc = fma(Qd[a * NX + j], y[a], acc);
          }
          z[j] = acc;
        }
      }
      // multipliers from z + N u = 0
#pragma unroll
      for (int a = MD - 1; a >= 0; --a) {
        double acc = -y[a];
#pragma unroll
        for (int l = a + 1; l < MD; ++l) {
          if (ad[l] != 0) acc = fma(-Rd[a * MD1 + l], ud[l], acc);
        }
        ud[a] = (ad[a] != 0) ? acc * iRd[a] : 0.0;
      }
      // equality rows with a negative multiplier are simply held from the other side
      bool flipped = false;
#pragma unroll
      for (int a = 0; a < MD; ++a) {
        uD[a] = ud[a];
        if (ad[a] != 0 && ud[a] < 0.0 && D.lbd[a] == D.ubd[a]) { ad[a] = -ad[a]; flipped = true; }
      }
      if (flipped) continue;                     // recompute with the new signs
      double worst = 0.0;
      int wi = -1;          // 0..NX-1 coordinate, NX.. dense slot
#pragma unroll
      for (int a = 0; a < MD; ++a) {
        if (ad[a] != 0 && ud[a] < worst) { worst = ud[a]; wi = NX + a; }
      }
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        if (nF[j] != 0.0) {
          double acc = z[j];
#pragma unroll
          for (int a = 0; a < MD; ++a) {
            if (ad[a] != 0) acc = fma((double)ad[a] * D.Ad[a * NX + j], ud[a], acc);
          }
          uF[j] = -acc * inF[j];
          if (uF[j] < worst) { worst = uF[j]; wi = j; }
        }
      }
      if (wi == -1) { warm_ok = true; break; }   // dual feasible: done
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        if (wi == j) { nF[j] = 0.0; inF[j] = 0.0; uF[j] = 0.0; frow[j] = -1; fside[j] = 0; z[j] = 0.0; }
      }
#pragma unroll
      for (int a = 0; a < MD; ++a) {
        if (wi == NX + a) { ad[a] = 0; uD[a] = 0.0; }
      }
      --nact;
    }
    if (!warm_ok) {                              // could not repair the guess: cold start
      nact = 0;
#pragma unroll
      for (int j = 0; j < NX; ++j) { z[j] = 0.0; nF[j] = 0.0; inF[j] = 0.0; uF[j] = 0.0; frow[j] = -1; fside[j] = 0; }
#pragma unroll
      for (int a = 0; a < MD; ++a) { ad[a] = 0; uD[a] = 0.0; }
    }
  }

  int status = QP_MAXITER;
  for (int it = 0; it < max_iter; ++it) {
    // ---- most violated one-sided constraint (same rule and tolerances as the dense solver) ----
    int p = -1;            // 0..MD-1: dense slot, MD..MD+MU-1: unit row
    double sp = 0.0, vbest = 0.0, bp = 0.0;   // bp: the violated bound, in the form n_p . z <= bp
#pragma unroll
    for (int a = 0; a < MD; ++a) {
      double r = 0.0;
#pragma unroll
      for (int j = 0; j < NX; ++j) r = fma(D.Ad[a * NX + j], z[j], r);
      const double vu = r - D.ubd[a], vl = D.lbd[a] - r;
      const double tu = 1e-12 * fmax(1.0, fabs(D.ubd[a])), tl = 1e-12 * fmax(1.0, fabs(D.lbd[a]));
      const bool free_ = ad[a] == 0;
      if (free_ && vu > tu && vu > vbest) { vbest = vu; p = a; sp = 1.0; bp = D.ubd[a]; }
      if (free_ && vl > tl && vl > vbest) { vbest = vl; p = a; sp = -1.0; bp = -D.lbd[a]; }
    }
#pragma unroll
    for (int i = 0; i < MU; ++i) {
      const double r = ks[i] * z[S::unit_col(i)];
      const double vu = r - D.ubu[i], vl = D.lbu[i] - r;
      const double tu = 1e-12 * fmax(1.0, fabs(D.ubu[i])), tl = 1e-12 * fmax(1.0, fabs(D.lbu[i]));
      const bool free_ = frow[S::unit_col(i)] != i;
      if (free_ && vu > tu && vu > vbest) { vbest = vu; p = MD + i; sp = 1.0; bp = D.ubu[i]; }
      if (free_ && vl > tl && vl > vbest) { vbest = vl; p = MD + i; sp = -1.0; bp = -D.lbu[i]; }
    }
    if (p < 0) { status = QP_OK; break; }

    // ---- its normal -------------------------------------------------------------------------------
    double np_[NX];
#pragma unroll
    for (int j = 0; j < NX; ++j) np_[j] = 0.0;
#pragma unroll
    for (int a = 0; a < MD; ++a) {
#pragma unroll
      for (int j = 0; j < NX; ++j) np_[j] = (p == a) ? sp * D.Ad[a * NX + j] : np_[j];
    }
#pragma unroll
    for (int i = 0; i < MU; ++i) {
      np_[S::unit_col(i)] = (p == MD + i) ? sp * ks[i] : np_[S::unit_col(i)];
    }
    double nn = 0.0, vnp = 1.0;
#pragma unroll
    for (int j = 0; j < NX; ++j) nn = fma(np_[j], np_[j], nn);
#pragma unroll
    for (int i = 0; i < MU; ++i) vnp = (p == MD + i) ? sp * ks[i] : vnp;

    double up = 0.0;
    bool done = false, infeasible = false;
    while (!done) {
      // ---- d = projection of n_p onto the null space of the working set, r = dual direction ------
      double d[NX], cd[MD1], rd[MD1], rF[NX];
#pragma unroll
      for (int j = 0; j < NX; ++j) d[j] = (nF[j] != 0.0) ? 0.0 : np_[j];
#pragma unroll
      for (int a = 0; a < MD; ++a) cd[a] = 0.0;
#pragma unroll
      for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
        for (int a = 0; a < MD; ++a) {           // inactive slots have Qd = 0: no-ops
          double dt = 0.0;
#pragma unroll
          for (int j = 0; j < NX; ++j) dt = fma(Qd[a * NX + j], d[j], dt);
#pragma unroll
          for (int j = 0; j < NX; ++j) d[j] = fma(-dt, Qd[a * NX + j], d[j]);
          cd[a] += dt;
        }
      }
#pragma unroll
      for (int a = MD - 1; a >= 0; --a) {
        double acc = cd[a];
#pragma unroll
        for (int l = a + 1; l < MD; ++l) acc = fma(-Rd[a * MD1 + l], rd[l], acc);
        rd[a] = acc * iRd[a];                      // iRd = 0 for an inactive slot
      }
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        double acc = np_[j];
#pragma unroll
        for (int a = 0; a < MD; ++a) acc = fma(-(double)ad[a] * D.Ad[a * NX + j], rd[a], acc);
        rF[j] = acc * inF[j];                      // inF = 0 for a free coordinate
      }
      double dn = 0.0;
#pragma unroll
      for (int j = 0; j < NX; ++j) dn = fma(d[j], d[j], dn);
      // ---- step lengths -----------------------------------------------------------------------------
      double rmax = 0.0;
#pragma unroll
      for (int j = 0; j < NX; ++j) rmax = fmax(rmax, fabs(rF[j]));
#pragma unroll
      for (int a = 0; a < MD; ++a) rmax = fmax(rmax, fabs(rd[a]));
      // ratio test min u/r over r > 0, compared by cross-multiplication (one division at the end)
      double ub_ = 0.0, rb_ = 0.0;
      int drop = -1;       // 0..NX-1: release coordinate, NX..NX+MD-1: dense slot
#pragma unroll
      for (int a = 0; a < MD; ++a) {
        if (ad[a] != 0 && rd[a] > 1e-12 * rmax && rd[a] > 0.0) {
          if (drop < 0 || uD[a] * rb_ < ub_ * rd[a]) { ub_ = uD[a]; rb_ = rd[a]; drop = NX + a; }
        }
      }
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        if (nF[j] != 0.0 && rF[j] > 1e-12 * rmax && rF[j] > 0.0) {
          if (drop < 0 || uF[j] * rb_ < ub_ * rF[j]) { ub_ = uF[j]; rb_ = rF[j]; drop = j; }
        }
      }
      const double t1 = (drop >= 0) ? ub_ / rb_ : INFINITY;
      double viol = -bp;                           // n_p . z - bound (> 0: violated)
#pragma unroll
      for (int j = 0; j < NX; ++j) viol = fma(np_[j], z[j], viol);
      const bool independent = (nact < NX) && (dn > 1e-24 * nn);
      const double t2 = independent ? viol / dn : INFINITY;
      const double t = fmin(t1, t2);
      if (!(t < INFINITY)) { infeasible = true; break; }
      if (independent) {
#pragma unroll
        for (int j = 0; j < NX; ++j) z[j] = fma(-t, d[j], z[j]);
      }
#pragma unroll
      for (int j = 0; j < NX; ++j) uF[j] = fma(-t, rF[j], uF[j]);
#pragma unroll
      for (int a = 0; a < MD; ++a) uD[a] = fma(-t, rd[a], uD[a]);
      up += t;
      if (t2 <= t1) {
        // full step: p joins the working set
#pragma unroll
        for (int a = 0; a < MD; ++a) {
          ad[a] = (p == a) ? ((sp > 0.0) ? 1 : -1) : ad[a];
          uD[a] = (p == a) ? up : uD[a];
        }
        const double inv_np = 1.0 / vnp;           // vnp: the single non-zero entry of a unit normal
#pragma unroll
        for (int i = 0; i < MU; ++i) {
          const bool hit = p == MD + i;
          nF[S::unit_col(i)] = hit ? vnp : nF[S::unit_col(i)];
          inF[S::unit_col(i)] = hit ? inv_np : inF[S::unit_col(i)];
          uF[S::unit_col(i)] = hit ? up : uF[S::unit_col(i)];
          frow[S::unit_col(i)] = hit ? i : frow[S::unit_col(i)];
          fside[S::unit_col(i)] = hit ? ((sp > 0.0) ? 1 : -1) : fside[S::unit_col(i)];
        }
        ++nact;
        done = true;
      } else {
        // partial step: release the blocking constraint, try again with the same p
#pragma unroll
        for (int j = 0; j < NX; ++j) {
          const bool hit = drop == j;
          nF[j] = hit ? 0.0 : nF[j];
          inF[j] = hit ? 0.0 : inF[j];
          uF[j] = hit ? 0.0 : uF[j];
          frow[j] = hit ? -1 : frow[j];
          fside[j] = hit ? 0 : fside[j];
        }
#pragma unroll
        for (int a = 0; a < MD; ++a) {
          ad[a] = (drop == NX + a) ? 0 : ad[a];
          uD[a] = (drop == NX + a) ? 0.0 : uD[a];
        }
        --nact;
      }
      refactor();
    }
    if (infeasible) { status = QP_INFEASIBLE; break; }
  }

#pragma unroll
  for (int j = 0; j < NX; ++j) x[j] = z[j] * D.s[j];
  unsigned mu = 0u, ml = 0u;
#pragma unroll
  for (int a = 0; a < MD; ++a) {
    if (S::dense_row(a) < 32) {
      if (ad[a] > 0) mu |= 1u << S::dense_row(a);
      if (ad[a] < 0) ml |= 1u << S::dense_row(a);
    }
  }
#pragma unroll
  for (int i = 0; i < MU; ++i) {
    if (S::unit_row(i) < 32 && frow[S::unit_col(i)] == i) {
      if (fside[S::unit_col(i)] > 0) mu |= 1u << S::unit_row(i); else ml |= 1u << S::unit_row(i);
    }
  }
  *act_up = mu;
  *act_lo = ml;
  return status;
}

// Working-set guess from a primal guess x0 (the reference's `x0=` warm start, reactive_qp.py:495-513):
// rows whose value at x0 sits on one of their bounds (relative 1e-9), plus every equality row.
template <class S>
__device__ __forceinline__ void masks_from_x0(const QpSData<S>& D, const double (&x0)[S::QN], unsigned* up,
                                              unsigned* lo) {
  unsigned mu = 0u, ml = 0u;
#pragma unroll
  for (int a = 0; a < S::QMD; ++a) {
    double r = 0.0;
#pragma unroll
    for (int j = 0; j < S::QN; ++j) r = fma(D.Ad[a * S::QN + j], x0[j], r);   // Ad still unscaled here
    if (S::dense_row(a) < 32) {
      if (D.lbd[a] == D.ubd[a] || fabs(r - D.ubd[a]) <= 1e-9 * (1.0 + fabs(D.ubd[a]))) mu |= 1u << S::dense_row(a);
      else if (fabs(r - D.lbd[a]) <= 1e-9 * (1.0 + fabs(D.lbd[a]))) ml |= 1u << S::dense_row(a);
    }
  }
#pragma unroll
  for (int i = 0; i < S::QMU; ++i) {
    const double r = S::unit_coef(i) * x0[S::unit_col(i)];
    if (S::unit_row(i) < 32) {
      if (fabs(r - D.ubu[i]) <= 1e-9 * (1.0 + fabs(D.ubu[i]))) mu |= 1u << S::unit_row(i);
      else if (fabs(r - D.lbu[i]) <= 1e-9 * (1.0 + fabs(D.lbu[i]))) ml |= 1u << S::unit_row(i);
    }
  }
  *up = mu;
  *lo = ml;
}

// Working-set guess when the caller has none ("crash start").  Goldfarb-Idnani adds one row per
// iteration, so a cold solve of the UR5 9x15 problem takes ~10 iterations and, worse, a warp runs for
// the maximum over its 32 instances (~15).  The guess is computed by a primal-dual active-set iteration
// (Hintermueller-Ito-Kunisch style): each pass solves "guessed dense rows held, guessed variables
// fixed at their bounds" exactly (a QMD x QMD Cholesky on the free variables), releases every held
// row / fixed variable whose multiplier has the wrong sign and takes up every row the face optimum
// violates (per variable the most violated
// row: joint position and joint speed limits bound the same column) — many rows change per pass, every
// thread does the same work, and the set is final when it stops changing (for that problem: 83 % of the
// instances after 3 passes, 99.4 % after 6).  Passes run until no thread of the warp changes its set
// (at most CRASH_PASSES; UR5 problem: 0.04 % of the instances are not final after 8 passes, 0.005 % after 12).  qp_structured then starts from the guess, repairs whatever is left and
// certifies the result, so the answer never depends on it.
constexpr int CRASH_PASSES = 12;
// MAXP: pass budget.  The fast pass of the two-launch form stops early (S::QP_FAST_PASSES): a warp runs
// until its SLOWEST lane is final, so with 32 instances per warp the average warp of the UR5 problem ran
// 6.2 passes although 83 % of the instances are final after 3 — the few slow ones are cheaper in the tail
// pass, which packs them densely and continues the passes from the parked set.
// SINGLE: apply only ONE of the changes a pass proposes (the most violated row if the face optimum is
// infeasible, else the held row with the worst multiplier).  The all-at-once passes can cycle between two
// sets (0.005 % of the UR5 instances never settle); changing one row at a time is the classical primal-dual
// pivoting rule and settles them, at one row per pass.  Used after the all-at-once budget is spent, in the
// kernels that hold the full solver anyway (never in the fast pass), so that almost nothing is left for
// the Goldfarb-Idnani iteration, whose single-thread latency (~30 us with its spills) was the whole
// duration of the tail launch.
constexpr int CRASH_SINGLE_PASSES = 30;
#ifdef CLIK_QP_STATS
static long long qp_pass_hist[2][64];   // host-harness instrumentation (tools/qp_pass_stats.py): passes per call [all-at-once / one-row]
#endif
template <class S, int MAXP = CRASH_PASSES, bool SINGLE = false>
__device__ __forceinline__ bool crash_guess(const QpSData<S>& D, unsigned* up /*in: guess, out*/,
                                            unsigned* lo, double (&xout)[S::QN], bool* still_changing = nullptr,
                                            const int passes_before = 0 /* passes an earlier launch spent on this set */) {
  constexpr int NX = S::QN, MD = S::QMD, MU = S::QMU, MD1 = MD > 0 ? MD : 1;
  bool eq[MD1];
  double s2[NX], yv[MD1];
  int fr[NX];                        // +(i+1) / -(i+1): variable fixed by unit row i at its upper / lower bound
  int da[MD1];                       // dense row held at its upper (+1) / lower (-1) bound, 0 = not held
  // the caller's guess (the previous step's working set in a rollout, or nothing) seeds the iteration:
  // an unchanged set is confirmed by the first pass
  const unsigned gu = *up, gl = *lo;
  // (the shortcut below for released variables is for cold predictions only: from a warm start — the
  // previous step's set in a rollout — a variable whose multiplier changes sign simply becomes free, and
  // testing it at its coordinate-wise optimum sends it to the opposite bound far too often: QP rollout
  // 6.9e9 -> 5.3e9 controller-steps/s with the shortcut applied to warm starts)
  const bool cold = (gu | gl) == 0u;
#pragma unroll
  for (int j = 0; j < NX; ++j) { s2[j] = D.s[j] * D.s[j]; fr[j] = 0; }
#pragma unroll
  for (int i = 0; i < MU; ++i) {
    const int c = S::unit_col(i);
    if (S::unit_row(i) < 32 && fr[c] == 0) {
      if (((gu >> S::unit_row(i)) & 1u) && fabs(D.ubu[i]) < INFINITY) fr[c] = i + 1;
      else if (((gl >> S::unit_row(i)) & 1u) && fabs(D.lbu[i]) < INFINITY) fr[c] = -(i + 1);
    }
  }
#pragma unroll
  for (int a = 0; a < MD; ++a) {
    eq[a] = (D.lbd[a] == D.ubd[a]) && (fabs(D.ubd[a]) < INFINITY) && S::dense_row(a) < 32;
    da[a] = eq[a] ? 1 : 0;
    if (S::dense_row(a) < 32 && !eq[a]) {
      if (((gu >> S::dense_row(a)) & 1u) && fabs(D.ubd[a]) < INFINITY) da[a] = 1;
      else if (((gl >> S::dense_row(a)) & 1u) && fabs(D.lbd[a]) < INFINITY) da[a] = -1;
    }
    yv[a] = 0.0;
  }
  bool certified = false;            // this thread's set stopped changing and its face optimum passes the KKT check
#pragma unroll 1
  for (int pass = 0; pass < MAXP; ++pass) {
    double xf[NX], w[NX];            // value of a fixed variable (0 if free); 1/h_j of a free one (0 if fixed)
#pragma unroll
    for (int j = 0; j < NX; ++j) xf[j] = 0.0;
#pragma unroll
    for (int i = 0; i < MU; ++i) {
      constexpr double one = 1.0;
      const double ik = one / S::unit_coef(i);
      const int c = S::unit_col(i);
      xf[c] = (fr[c] == i + 1) ? D.ubu[i] * ik : ((fr[c] == -(i + 1)) ? D.lbu[i] * ik : xf[c]);
    }
#pragma unroll
    for (int j = 0; j < NX; ++j) w[j] = (fr[j] == 0) ? s2[j] : 0.0;
    // equality rows restricted to the free variables: Gram matrix and right-hand side (Ad is unscaled here)
    double G[MD1 * MD1];
#pragma unroll
    for (int a = 0; a < MD; ++a) {
      double rhs = (da[a] < 0) ? D.lbd[a] : D.ubd[a];
#pragma unroll
      for (int j = 0; j < NX; ++j) { if (S::ad_nz(a, j)) rhs = fma(-D.Ad[a * NX + j], xf[j], rhs); }
      yv[a] = (da[a] != 0) ? rhs : 0.0;
#pragma unroll
      for (int b = 0; b <= a; ++b) {
        double g = 0.0;
#pragma unroll
        for (int j = 0; j < NX; ++j) { if (S::ad_nz(a, j) && S::ad_nz(b, j)) g = fma(D.Ad[a * NX + j] * w[j], D.Ad[b * NX + j], g); }
        G[a * MD1 + b] = (da[a] != 0 && da[b] != 0) ? g : ((a == b) ? 1.0 : 0.0);
      }
    }
    // Cholesky G = L L' (a numerically dependent row drops out: its pivot inverse is 0), y = G^-1 rhs
    double dinv[MD1];
#pragma unroll
    for (int a = 0; a < MD; ++a) {
      double dg = G[a * MD1 + a];
      const double scale = dg;
#pragma unroll
      for (int k = 0; k < a; ++k) dg = fma(-G[a * MD1 + k], G[a * MD1 + k], dg);
      dinv[a] = (dg > 1e-12 * scale) ? rsqrt(dg) : 0.0;
#pragma unroll
      for (int b = a + 1; b < MD; ++b) {
        double v = G[b * MD1 + a];
#pragma unroll
        for (int k = 0; k < a; ++k) v = fma(-G[b * MD1 + k], G[a * MD1 + k], v);
        G[b * MD1 + a] = v * dinv[a];
      }
    }
#pragma unroll
    for (int a = 0; a < MD; ++a) {
      double v = yv[a];
#pragma unroll
      for (int k = 0; k < a; ++k) v = fma(-G[a * MD1 + k], yv[k], v);
      yv[a] = v * dinv[a];
    }
#pragma unroll
    for (int a = MD - 1; a >= 0; --a) {
      double v = yv[a];
#pragma unroll
      for (int k = a + 1; k < MD; ++k) v = fma(-G[k * MD1 + a], yv[k], v);
      yv[a] = v * dinv[a];
    }
    // face optimum: a free variable sits at xfree = (A_eq' y)_j / h_j; a fixed one keeps its bound and
    // has a multiplier of the sign of (bound - xfree) / coefficient
    double xc[NX], gs[NX], viol[NX];
    int nf[NX];
#pragma unroll
    for (int j = 0; j < NX; ++j) {
      double tj = 0.0;
#pragma unroll
      for (int a = 0; a < MD; ++a) { if (S::ad_nz(a, j)) tj = fma(D.Ad[a * NX + j], yv[a], tj); }
      const double xfree = s2[j] * tj;
      xc[j] = (fr[j] == 0) ? xfree : xf[j];
      gs[j] = xf[j] - xfree;
      nf[j] = 0;
      viol[j] = 0.0;
    }
#pragma unroll
    for (int i = 0; i < MU; ++i) {
      const int c = S::unit_col(i);
      const double gk = gs[c] * S::unit_coef(i);
      nf[c] = (fr[c] == i + 1 && gk <= 0.0) ? i + 1 : ((fr[c] == -(i + 1) && gk >= 0.0) ? -(i + 1) : nf[c]);
    }
    // A fixed variable whose multiplier has the wrong sign is released — and in the first passes tested at
    // the value it would take if it were free with the dense multipliers as they are (xfree): when that lies
    // beyond one of its bounds (typically the opposite one: the first pass clamps every joint at the sign of
    // the unconstrained optimum, and a far target turns some of them around) the variable moves to that bound
    // in this pass instead of going through "free" first.  For the UR5 problem this takes the mean number
    // of passes from 3.6 to 2.8 and the share of instances final after 3 passes from 40 % to 91 %
    // (profiles/r2_qp_pass_stats.txt).  Only a guess changes: every set is still certified by a pass that
    // leaves it unchanged.  Later passes release to "free" (a two-bound flip-flop cannot form), and so do
    // all passes of a warm-started prediction.
    double xt[NX];
    const bool flip = !SINGLE && cold && passes_before + pass < S::QP_FLIP_PASSES;
#pragma unroll
    for (int j = 0; j < NX; ++j) xt[j] = (flip && fr[j] != 0 && nf[j] == 0) ? xc[j] - gs[j] : xc[j];
#pragma unroll
    for (int i = 0; i < MU; ++i) {
      constexpr double one = 1.0;
      const int c = S::unit_col(i);
      const double ik = one / (S::unit_coef(i) < 0.0 ? -S::unit_coef(i) : S::unit_coef(i));
      const double r = S::unit_coef(i) * xt[c];
      const double vu = (r - D.ubu[i]) * ik, vl = (D.lbu[i] - r) * ik;
      if (S::unit_row(i) < 32) {
        if (vu > 1e-12 * fmax(1.0, fabs(D.ubu[i])) * ik && vu > viol[c]) { viol[c] = vu; nf[c] = i + 1; }
        if (vl > 1e-12 * fmax(1.0, fabs(D.lbu[i])) * ik && vl > viol[c]) { viol[c] = vl; nf[c] = -(i + 1); }
      }
    }
    bool changed = false;
#pragma unroll
    for (int j = 0; j < NX; ++j) changed = changed || (nf[j] != fr[j]);
    // dense inequality rows: keep while the multiplier (-y for upper, +y for lower) is non-negative,
    // take up when the face optimum violates them (equality rows always stay)
    bool held_ok = true;             // every held dense row really sits on its bound (the Gram solve was accurate)
    int nd[MD1];
    double dviol[MD1];
#pragma unroll
    for (int a = 0; a < MD; ++a) {
      double r = 0.0;
#pragma unroll
      for (int j = 0; j < NX; ++j) { if (S::ad_nz(a, j)) r = fma(D.Ad[a * NX + j], xc[j], r); }
      const double bnd = (da[a] < 0) ? D.lbd[a] : D.ubd[a];
      held_ok = held_ok && (da[a] == 0 || fabs(r - bnd) <= 1e-11 * (1.0 + fabs(bnd)));
      int na = (da[a] > 0 && yv[a] <= 0.0) ? 1 : ((da[a] < 0 && yv[a] >= 0.0) ? -1 : 0);
      if (da[a] == 0 && S::dense_row(a) < 32) {
        if (r - D.ubd[a] > 1e-12 * fmax(1.0, fabs(D.ubd[a]))) na = 1;
        if (D.lbd[a] - r > 1e-12 * fmax(1.0, fabs(D.lbd[a]))) na = -1;
      }
      na = eq[a] ? 1 : na;
      changed = changed || (na != da[a]);
      nd[a] = na;
      dviol[a] = fmax(r - D.ubd[a], D.lbd[a] - r);
    }
    if constexpr (SINGLE) {
      double best = 0.0;
      int pick = -1;                   // 0..NX-1: variable, NX..: dense row
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        if (nf[j] != fr[j] && viol[j] > best) { best = viol[j]; pick = j; }
      }
#pragma unroll
      for (int a = 0; a < MD; ++a) {
        if (nd[a] != da[a] && da[a] == 0 && dviol[a] > best) { best = dviol[a]; pick = NX + a; }
      }
      if (pick < 0) {                  // primal feasible: release the worst multiplier
#pragma unroll
        for (int j = 0; j < NX; ++j) {
          if (nf[j] != fr[j] && fabs(gs[j]) >= best) { best = fabs(gs[j]); pick = j; }
        }
#pragma unroll
        for (int a = 0; a < MD; ++a) {
          if (nd[a] != da[a] && fabs(yv[a]) >= best) { best = fabs(yv[a]); pick = NX + a; }
        }
      }
#pragma unroll
      for (int j = 0; j < NX; ++j) fr[j] = (pick == j) ? nf[j] : fr[j];
#pragma unroll
      for (int a = 0; a < MD; ++a) da[a] = (pick == NX + a) ? nd[a] : da[a];
    } else {
#pragma unroll
      for (int j = 0; j < NX; ++j) fr[j] = nf[j];
#pragma unroll
      for (int a = 0; a < MD; ++a) da[a] = nd[a];
    }
    // unchanged set = every row feasible, every multiplier of the right sign: the face optimum is the
    // minimiser.  (A later pass of a thread that waits for its warp recomputes the same numbers.)
    certified = !changed && held_ok;
    // (a set that stopped changing without certifying — an inaccurate Gram solve near a singular task
    // Jacobian — will not be helped by more passes: the caller goes straight to the iteration)
    if (still_changing != nullptr) *still_changing = changed;
#pragma unroll
    for (int j = 0; j < NX; ++j) xout[j] = xc[j];
#ifdef CLIK_QP_STATS
    if (!changed || pass == MAXP - 1) ++qp_pass_hist[SINGLE ? 1 : 0][pass + 1 < 64 ? pass + 1 : 63];
#endif
    if (!__any_sync(__activemask(), changed)) break;
  }
  unsigned mu = 0u, ml = 0u;
  // an equality row is held from the side that gives it a non-negative multiplier (u = -+y)
#pragma unroll
  for (int a = 0; a < MD; ++a) {
    if (eq[a]) {
      if (yv[a] > 0.0) ml |= 1u << S::dense_row(a); else mu |= 1u << S::dense_row(a);
    } else if (da[a] != 0) {
      if (da[a] > 0) mu |= 1u << S::dense_row(a); else ml |= 1u << S::dense_row(a);
    }
  }
#pragma unroll
  for (int i = 0; i < MU; ++i) {
    if (fr[S::unit_col(i)] == i + 1) mu |= 1u << S::unit_row(i);
    if (fr[S::unit_col(i)] == -(i + 1)) ml |= 1u << S::unit_row(i);
  }
  *up = mu;
  *lo = ml;
  return certified;
}

// Everything S::eval_qp produces for one instance.
template <class S> struct QpData {
  double A[S::QM * S::QN];
  double lb[S::QM];
  double ub[S::QM];
  double h[S::QN];
};

// One instance of the fused step: load, evaluate the skill's QP matrices, solve, store.
// MODE QP_FAST: the first S::QP_FAST_PASSES prediction passes; an instance they cannot certify is marked
// QP_PENDING in status[i], its uncertified set is parked in active[] (if present), nothing else is written.
// MODE QP_TAIL: such an instance, packed densely with the other slow ones: the rest of the all-at-once
// budget and the one-row passes from the parked set, then the Goldfarb-Idnani iteration for what is still
// uncertified (the whole path when there is no active[] to park in).  MODE QP_FULL: everything, one thread.
// FAST -> TAIL run exactly the pass sequence of FULL, hence the same bits.
enum : int { QP_FULL = 0, QP_FAST = 1, QP_TAIL = 2 };
#ifdef CLIK_QP_STATS
static long long qp_stats[8];   // host-harness instrumentation: [0] instances entering Goldfarb-Idnani, [1] one-row phases
#endif
template <class S, int MODE>
__device__ __forceinline__ void qp_instance(long long ld, long long i, const double* __restrict__ t, int t_stride,
                                            const double* __restrict__ q, const double* __restrict__ x,
                                            const double* __restrict__ y, const double* __restrict__ x0,
                                            const unsigned* active0, double* __restrict__ sol,
                                            int* __restrict__ status, unsigned* active, int max_iter) {
  double qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
  // only the rows the generated program reads are fetched and tested (S::QP_READ_*): an unread row may
  // be anything — the host entry points do not even upload it
  const double tv = S::QP_READ_T ? __ldcs(t + (long long)t_stride * i) : 0.0;
  bool data_ok = finite_bits(tv);
#pragma unroll
  for (int j = 0; j < S::NQ; ++j) {
    qv[j] = row_read(S::QP_READ_Q, j) ? __ldcs(q + (long long)j * ld + i) : 0.0;
    data_ok = data_ok && finite_bits(qv[j]);
  }
#pragma unroll
  for (int j = 0; j < S::NX; ++j) {
    xv[j] = row_read(S::QP_READ_X, j) ? __ldcs(x + (long long)j * ld + i) : 0.0;
    data_ok = data_ok && finite_bits(xv[j]);
  }
#pragma unroll
  for (int j = 0; j < S::NY; ++j) {
    yv[j] = row_read(S::QP_READ_Y, j) ? __ldcs(y + (long long)j * ld + i) : 0.0;
    data_ok = data_ok && finite_bits(yv[j]);
  }
  double xs[S::QN];
  unsigned mu = 0u, ml = 0u;
  int st;
  if constexpr (S::QSTRUCT) {
    QpSData<S> d;
    S::eval_qps(tv, qv, xv, yv, d);
    // warm start: an explicit working-set guess (active0, may alias `active`) wins over one
    // derived from the primal guess x0; neither changes the answer, only the iteration count
    unsigned wu = 0u, wl = 0u;
    const bool parked = MODE == QP_TAIL && active != nullptr;
    if (parked) {
      wu = active[i];
      wl = active[ld + i];
    } else if (active0 != nullptr) {
      wu = active0[i];
      wl = active0[ld + i];
    } else if (x0 != nullptr) {
      double x0v[S::QN];
#pragma unroll
      for (int j = 0; j < S::QN; ++j) x0v[j] = x0[(long long)j * ld + i];
      masks_from_x0<S>(d, x0v, &wu, &wl);
    } else if (!S::QP_CRASH && S::QP_EQ_START) {
      // no guess: equality rows are active at every solution, start with them held
#pragma unroll
      for (int a = 0; a < S::QMD; ++a) {
        if (S::dense_row(a) < 32 && d.lbd[a] == d.ubd[a]) wu |= 1u << S::dense_row(a);
      }
    }
    // predicts the working set from any guess, or none; when the prediction certifies itself its
    // face optimum is the answer and the iteration below is skipped
    constexpr int REST = CRASH_PASSES - S::QP_FAST_PASSES > 1 ? CRASH_PASSES - S::QP_FAST_PASSES : 1;
    bool ok = false;
    if constexpr (MODE == QP_FAST) {
      if (S::QP_CRASH) ok = crash_guess<S, S::QP_FAST_PASSES>(d, &wu, &wl, xs);
    } else {
      if (S::QP_CRASH) {
        bool cycling = false;
        ok = parked ? crash_guess<S, REST>(d, &wu, &wl, xs, &cycling, S::QP_FAST_PASSES)   // same pass sequence as QP_FULL
                    : crash_guess<S>(d, &wu, &wl, xs, &cycling);
        if (!ok && cycling && S::QP_CRASH_SINGLE) {
#ifdef CLIK_QP_STATS
          ++qp_stats[1];
#endif
          ok = crash_guess<S, CRASH_SINGLE_PASSES, true>(d, &wu, &wl, xs);
        }
      }
    }
    const bool solved = ok && S::QP_CRASH_FINAL && all_finite(xs) && data_ok;
    st = solved ? QP_OK : QP_MAXITER;
    mu = wu;
    ml = wl;
    if constexpr (MODE == QP_FAST) {
      if (!solved && data_ok) {
        status[i] = QP_PENDING;
        if (active != nullptr) {
          active[i] = wu;
          active[ld + i] = wl;
        }
        return;
      }
    } else {
#ifdef CLIK_QP_STATS
      if (!solved && data_ok) ++qp_stats[0];
#endif
#pragma unroll 1
      for (int attempt = 0; attempt < 2 && !solved && data_ok; ++attempt) {   // a bad guess must never cost the answer:
        if (attempt > 0) {                                         // second attempt = cold start
          wu = wl = 0u;
          S::eval_qps(tv, qv, xv, yv, d);
        }
        st = qp_structured<S>(d, xs, &mu, &ml, max_iter, wu, wl);
        if (st == QP_OK || (wu | wl) == 0u) break;
      }
    }
  } else {
    QpData<S> d;
    S::eval_qp(tv, qv, xv, yv, d);
    st = qp_dual_active_set<S::QN, S::QM>(S::QN, S::QM, d.A, d.lb, d.ub, d.h, nullptr, xs, &mu, &ml,
                                          max_iter);
  }
  // NaN / inf in the inputs or in the solution is never "solved": the iteration sees every comparison
  // with a NaN as false and would report the start point as optimal
  if (!data_ok || (st == QP_OK && !all_finite(xs))) {
    st = QP_INVALID;
    mu = ml = 0u;
  }
  for (int j = 0; j < S::QN; ++j) __stcs(sol + (long long)j * ld + i, xs[j]);
  if (status != nullptr) status[i] = st;
  if (active != nullptr) {
    active[i] = mu;
    active[ld + i] = ml;
  }
}

// Fused step, SoA in / SoA out: sol[j*ld + i] is entry j of x for instance i; active[i] = upper mask,
// active[ld + i] = lower mask (N instances, row stride ld >= N: see pinv_step).  One kernel does everything (MODE = QP_FULL), or — structured skills with
// the working-set prediction, status array present — a QP_FAST pass followed by qp_step_tail.  The split
// keeps the Goldfarb-Idnani iteration (255 registers + spills, needed by well under 1 % of the
// instances) out of the kernel every instance runs (159 registers for the UR5 problem).
template <class S, int MODE>
__device__ __forceinline__ void qp_step(long long N, long long ld, const double* __restrict__ t, int t_stride,
                                        const double* __restrict__ q, const double* __restrict__ x,
                                        const double* __restrict__ y, const double* __restrict__ x0,
                                        const unsigned* active0, double* __restrict__ sol,
                                        int* __restrict__ status, unsigned* active, int max_iter) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride)
    qp_instance<S, MODE>(ld, i, t, t_stride, q, x, y, x0, active0, sol, status, active, max_iter);
}

// Tail pass: every CTA scans QP_TAIL_TILE consecutive status entries, collects the instances the FAST
// pass left QP_PENDING into shared memory and solves those with the full path, densely packed into
// its first threads (no global scratch, so calls on different streams do not interfere).
constexpr int QP_TAIL_TILE = 1024;
#ifdef __CUDACC__   // (the host-compiled test harness of the solvers has no shared memory)
template <class S>
__device__ __forceinline__ void qp_step_tail(long long N, long long ld, const double* __restrict__ t, int t_stride,
                                             const double* __restrict__ q, const double* __restrict__ x,
                                             const double* __restrict__ y, const double* __restrict__ x0,
                                             const unsigned* active0, double* __restrict__ sol,
                                             int* __restrict__ status, unsigned* active, int max_iter) {
  __shared__ int list[QP_TAIL_TILE];
  __shared__ int count;
  for (long long base = (long long)blockIdx.x * QP_TAIL_TILE; base < N; base += (long long)gridDim.x * QP_TAIL_TILE) {
    if (threadIdx.x == 0) count = 0;
    __syncthreads();
    for (int k = threadIdx.x; k < QP_TAIL_TILE && base + k < N; k += blockDim.x) {
      if (status[base + k] == QP_PENDING) list[atomicAdd(&count, 1)] = k;
    }
    __syncthreads();
    const int n = count;
    for (int k = threadIdx.x; k < n; k += blockDim.x)
      qp_instance<S, QP_TAIL>(ld, base + list[k], t, t_stride, q, x, y, x0, active0, sol, status, active, max_iter);
    __syncthreads();
  }
}

#endif

// One step of the closed-loop rollouts (qp_rollout and the tangent rollouts of clik_jvp.cuh): the QP at
// (tv, qv, xv, yv), started from the working set (mu, ml) of the previous step, which it replaces.  Returns the
// status (QP_INVALID for a non-finite solution); xs = the unclipped solution.
template <class S>
__device__ __forceinline__ int qp_rollout_solve(double tv, const double (&qv)[S::NQ > 0 ? S::NQ : 1],
                                                const double (&xv)[S::NX > 0 ? S::NX : 1],
                                                const double (&yv)[S::NY > 0 ? S::NY : 1], double (&xs)[S::QN],
                                                unsigned& mu, unsigned& ml, int max_iter) {
  int st;
  if constexpr (S::QSTRUCT) {
    QpSData<S> d;
    S::eval_qps(tv, qv, xv, yv, d);
    unsigned wu = mu, wl = ml;
    bool solved = false;            // previous step's set -> this step's (usually one pass)
    if (S::QP_CRASH) {
      bool cycling = false;
      bool ok = crash_guess<S>(d, &wu, &wl, xs, &cycling);
      if (!ok && cycling && S::QP_CRASH_SINGLE) ok = crash_guess<S, CRASH_SINGLE_PASSES, true>(d, &wu, &wl, xs);
      solved = ok && S::QP_CRASH_FINAL && all_finite(xs);
    }
    st = solved ? QP_OK : QP_MAXITER;
    if (solved) { mu = wu; ml = wl; }
#pragma unroll 1
    for (int attempt = 0; attempt < 2 && !solved; ++attempt) {
      if (attempt > 0) {
        wu = wl = 0u;
        S::eval_qps(tv, qv, xv, yv, d);
      }
      st = qp_structured<S>(d, xs, &mu, &ml, max_iter, wu, wl);
      if (st == QP_OK || (wu | wl) == 0u) break;
    }
  } else {
    QpData<S> d;
    S::eval_qp(tv, qv, xv, yv, d);
    st = qp_dual_active_set<S::QN, S::QM>(S::QN, S::QM, d.A, d.lb, d.ub, d.h, nullptr, xs, &mu, &ml,
                                          max_iter);
  }
  if (st == QP_OK && !all_finite(xs)) st = QP_INVALID;
  return st;
}

// The clip and the Euler update of a rollout step (QP and NLP): v = clip(xs[:n], +-max_speed) in place,
// q += v_rob*dt, x += v_virt*dt.
template <class S, int NN>
__device__ __forceinline__ void rollout_euler(double (&xs)[NN], double (&qv)[S::NQ > 0 ? S::NQ : 1],
                                              double (&xv)[S::NX > 0 ? S::NX : 1], double vmax_q, double vmax_x,
                                              double dt) {
  for (int j = 0; j < S::NQ; ++j) {
    xs[j] = fmax(fmin(xs[j], vmax_q), -vmax_q);
    qv[j] = __dadd_rn(qv[j], __dmul_rn(xs[j], dt));
  }
  for (int j = 0; j < S::NX; ++j) {
    xs[S::NQ + j] = fmax(fmin(xs[S::NQ + j], vmax_x), -vmax_x);
    xv[j] = __dadd_rn(xv[j], __dmul_rn(xs[S::NQ + j], dt));
  }
}

// Applies a solved QP rollout step: an unsolved one (st != QP_OK) applies zero velocity and is counted in failed;
// xs is left clipped, the next step's start.
template <class S>
__device__ __forceinline__ void qp_rollout_advance(int st, double (&xs)[S::QN], double (&qv)[S::NQ > 0 ? S::NQ : 1],
                                                   double (&xv)[S::NX > 0 ? S::NX : 1], double vmax_q,
                                                   double vmax_x, double dt, int& failed) {
  if (st != QP_OK) {
    ++failed;
    for (int j = 0; j < S::QN; ++j) xs[j] = 0.0;
  }
  rollout_euler<S>(xs, qv, xv, vmax_q, vmax_x, dt);
}

// Closed-loop rollout with the QP controller: `steps` times  sol = solve(t0 + k*dt, q, x, y);
// v = clip(sol[:n], +-max_speed); q += v_rob*dt; x += v_virt*dt  (the notebooks' simulation loop,
// ur5_moe2016_example2.ipynb cell 12).  A step whose QP is not solved (status != 0; the reference
// would raise there) applies zero velocity and is counted in n_failed.
template <class S>
__device__ __forceinline__ void qp_rollout(long long N, long long ld, int steps, double dt, const double* __restrict__ t0,
                                           int t_stride, double* __restrict__ q, double* __restrict__ x,
                                           const double* __restrict__ y, double vmax_q, double vmax_x,
                                           double* __restrict__ sol_last, int* __restrict__ n_failed,
                                           int max_iter) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    double qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
    const double t0v = t0[(long long)t_stride * i];
    for (int j = 0; j < S::NQ; ++j) qv[j] = q[(long long)j * ld + i];
    for (int j = 0; j < S::NX; ++j) xv[j] = x[(long long)j * ld + i];
    for (int j = 0; j < S::NY; ++j) yv[j] = y[(long long)j * ld + i];
    double xs[S::QN];
    for (int j = 0; j < S::QN; ++j) xs[j] = 0.0;
    int failed = 0;
    unsigned mu = 0u, ml = 0u;        // working set of the previous step = warm start of the next
    for (int k = 0; k < steps; ++k) {
      const double tv = __dadd_rn(t0v, __dmul_rn(dt, (double)k));
      const int st = qp_rollout_solve<S>(tv, qv, xv, yv, xs, mu, ml, max_iter);
      qp_rollout_advance<S>(st, xs, qv, xv, vmax_q, vmax_x, dt, failed);
    }
    for (int j = 0; j < S::NQ; ++j) q[(long long)j * ld + i] = qv[j];
    for (int j = 0; j < S::NX; ++j) x[(long long)j * ld + i] = xv[j];
    if (sol_last != nullptr)
      for (int j = 0; j < S::QN; ++j) sol_last[(long long)j * ld + i] = xs[j];
    if (n_failed != nullptr) n_failed[i] = failed;
  }
}

}  // namespace clik
