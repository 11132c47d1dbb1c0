// clik_nlp.cuh — batched reactive-NLP controller step, one instance per thread, fp64, sm_100a.
//
//     min F(x) = cost(t, q, x, y; x_dec) + slack' diag(mu + w_slack) slack     s.t.  lb <= A x <= ub
//
// over x = [robot vel; virtual vel; slack], with A, lb, ub exactly the rows of the reactive QP
// (clik_qp.cuh).  The constraints are linear in the decision variables, so the problem is a linearly
// constrained NLP of fixed shape; it is solved by sequential quadratic programming with the exact
// Hessian.  Each subproblem
//
//     min 1/2 p' B p + g' p,   lb - A v <= A p <= ub - A v,     B = H + delta I = L L'
//
// is reduced to the least-distance form the dense QP core solves (qp_dual_active_set with h = 1):
// with u = L' p + w, w = L^-1 g, the objective is 1/2 |u|^2 - const and the rows become
// A' = A L^-T with bounds shifted by A' w; then p = L^-T (u - w).  The first step is a full step (it
// restores feasibility from the start point); after that every iterate is feasible and the feasible set
// is convex, so a backtracking Armijo search on F alone keeps feasibility.  A cost whose Hessian does not
// depend on the decision variables (S::NLP_QUADRATIC) and needs no shift is solved by its first subproblem.
//
// Stop when |p|_inf * max(1, delta) <= tol * (1 + |v|_inf), or when a step with
// |p|_inf <= NLP_FLOOR_STEP * tol * (1 + |v|_inf) leaves F unchanged within its rounding
// (|dF| <= NLP_F_FLOOR * |F|): the subproblem's own accuracy can keep |p| a few tol above tol.
//
// The generated skill provides (codegen/emit.py):
//   S::NN, S::NM, S::NP        decision variables, constraint rows, hoisted decision-free values
//   S::eval_nlp_pre(t,q,x,y,d) A, lb, ub and P (forward kinematics, Jacobian entries, weights ...) once per step
//   S::eval_nlp_f(P, v)        F at v
//   S::eval_nlp_fgH(P, v, g, H) F, gradient and packed lower Hessian (H[i*(i+1)/2 + j], j <= i) at v
//   S::NLP_TOL, S::NLP_QP_ITER stopping tolerance, iteration cap of each subproblem
#pragma once
#include <cmath>

#include "clik_qp.cuh"

namespace clik {

enum : int { NLP_OK = 0, NLP_MAXITER = 1, NLP_INFEASIBLE = 2, NLP_INVALID = 4, NLP_STALLED = 5 };

constexpr int NLP_REG_TRIES = 10;    // Hessian shifts tried: 1e-8 .. 1e10 times max(1, max |H_jj|)
constexpr int NLP_LS_TRIES = 40;     // Armijo halvings before the step is declared stalled
constexpr double NLP_ARMIJO_C1 = 1e-4;
constexpr double NLP_F_FLOOR = 1e-15;    // change of F within its rounding: |dF| <= 1e-15 |F| (+ NLP_F_ABS) ...
constexpr double NLP_F_ABS = 1e-300;     //   (absolute term: F = 0 exactly)
constexpr double NLP_FLOOR_STEP = 1e2;    // ... by a step within this factor of the tolerance

template <class S> struct NlpData {
  double A[S::NM * S::NN];
  double lb[S::NM], ub[S::NM];
  double P[S::NP > 0 ? S::NP : 1];
};

// B = H + delta I = L L' (both packed lower); false when a pivot is <= piv
template <int N>
__device__ __forceinline__ bool nlp_cholesky(const double* H, double delta, double piv, double* L) {
  for (int j = 0; j < N; ++j) {
    const int jj = j * (j + 1) / 2;
    double s = H[jj + j] + delta;
    for (int k = 0; k < j; ++k) s = fma(-L[jj + k], L[jj + k], s);
    if (!(s > piv)) return false;
    const double ljj = sqrt(s);
    L[jj + j] = ljj;
    const double inv = 1.0 / ljj;
    for (int i = j + 1; i < N; ++i) {
      const int ii = i * (i + 1) / 2;
      double a = H[ii + j];
      for (int k = 0; k < j; ++k) a = fma(-L[ii + k], L[jj + k], a);
      L[ii + j] = a * inv;
    }
  }
  return true;
}

// b <- L^-1 b
template <int N>
__device__ __forceinline__ void nlp_lsolve(const double* L, double* b) {
  for (int i = 0; i < N; ++i) {
    const int ii = i * (i + 1) / 2;
    double a = b[i];
    for (int k = 0; k < i; ++k) a = fma(-L[ii + k], b[k], a);
    b[i] = a / L[ii + i];
  }
}

// b <- L^-T b
template <int N>
__device__ __forceinline__ void nlp_ltsolve(const double* L, double* b) {
  for (int i = N - 1; i >= 0; --i) {
    double a = b[i];
    for (int k = i + 1; k < N; ++k) a = fma(-L[k * (k + 1) / 2 + i], b[k], a);
    b[i] = a / L[i * (i + 1) / 2 + i];
  }
}

template <int N>
__device__ __forceinline__ double nlp_norm_inf(const double* a) {
  double r = 0.0;
  for (int j = 0; j < N; ++j) r = fmax(r, fabs(a[j]));
  return r;
}

// One instance: d evaluated by S::eval_nlp_pre, v = start point on entry (x0 or 0), solution on return.
// Returns NLP_*; *iters = SQP iterations (subproblems solved), act_up / act_lo = working set of the last
// subproblem in the QP controller's mask format.
template <class S>
__device__ __noinline__ int nlp_solve(NlpData<S>& d, double (&v)[S::NN], unsigned* act_up, unsigned* act_lo,
                                      int* iters, const int max_iter) {
  constexpr int N = S::NN, M = S::NM, NH = S::NN * (S::NN + 1) / 2;
  constexpr int M1 = M > 0 ? M : 1;
  double g[N], H[NH], L[NH], w[N], z[N], p[N], one[N], vt[N];
  double Ap[M1 * N], lbp[M1], ubp[M1];
  *act_up = 0u;
  *act_lo = 0u;
  *iters = 0;
  // problem data: A and P finite, bounds not NaN (+-inf bounds are allowed)
  bool ok = true;
  for (int k = 0; k < M * N; ++k) ok = ok && finite_bits(d.A[k]);
  for (int r = 0; r < M; ++r) ok = ok && !(d.lb[r] != d.lb[r]) && !(d.ub[r] != d.ub[r]);
  for (int k = 0; k < S::NP; ++k) ok = ok && finite_bits(d.P[k]);
  if (!ok) return NLP_INVALID;
  for (int j = 0; j < N; ++j) one[j] = 1.0;
  int status = NLP_MAXITER;
  for (int it = 0; it < max_iter; ++it) {
    const double F0 = S::eval_nlp_fgH(d.P, v, g, H);
    bool fin = finite_bits(F0);
    for (int j = 0; j < N; ++j) fin = fin && finite_bits(g[j]) && finite_bits(v[j]);
    for (int k = 0; k < NH; ++k) fin = fin && finite_bits(H[k]);
    if (!fin) { status = NLP_INVALID; break; }
    // ---- B = H + delta I = L L' ------------------------------------------------------------------
    double hmax = 1.0;
    for (int j = 0; j < N; ++j) hmax = fmax(hmax, fabs(H[j * (j + 1) / 2 + j]));
    const double piv = 1e-12 * hmax;
    double shift = 0.0;
    bool factored = nlp_cholesky<N>(H, 0.0, piv, L);
    for (int k = 0; k < NLP_REG_TRIES && !factored; ++k) {
      shift = (k == 0) ? 1e-8 * hmax : shift * 100.0;
      factored = nlp_cholesky<N>(H, shift, piv, L);
    }
    if (!factored) { status = NLP_INVALID; break; }
    // ---- least-distance subproblem: rows A' = A L^-T, bounds shifted by A' w - A v ------------------
    for (int j = 0; j < N; ++j) w[j] = g[j];
    nlp_lsolve<N>(L, w);
    for (int r = 0; r < M; ++r) {
      double* row = &Ap[r * N];
      double av = 0.0;
      for (int j = 0; j < N; ++j) { row[j] = d.A[r * N + j]; av = fma(row[j], v[j], av); }
      nlp_lsolve<N>(L, row);   // (A L^-T)_r = (L^-1 a_r)'
      double aw = 0.0;
      for (int j = 0; j < N; ++j) aw = fma(row[j], w[j], aw);
      lbp[r] = d.lb[r] - av + aw;
      ubp[r] = d.ub[r] - av + aw;
    }
    unsigned mu = 0u, ml = 0u;
    const int qst = qp_dual_active_set<N, M1>(N, M, Ap, lbp, ubp, one, nullptr, z, &mu, &ml, S::NLP_QP_ITER);
    *iters = it + 1;
    *act_up = mu;
    *act_lo = ml;
    if (qst == QP_INFEASIBLE) { status = NLP_INFEASIBLE; break; }
    if (qst != QP_OK) { status = NLP_MAXITER; break; }
    for (int j = 0; j < N; ++j) p[j] = z[j] - w[j];
    nlp_ltsolve<N>(L, p);
    // a vanishing step is a stationary point of F when B = H (with a shift, the step shrinks with it: the
    // residual of stationarity is B p, hence the factor); a convex quadratic cost is solved by one step
    const bool converged = nlp_norm_inf<N>(p) * fmax(1.0, shift) <= S::NLP_TOL * (1.0 + nlp_norm_inf<N>(v));
    const bool exact = S::NLP_QUADRATIC && shift == 0.0;
    if (it == 0 || exact || converged) {
      // first step (restores feasibility from the start point), the answer, or a vanishing step
      for (int j = 0; j < N; ++j) v[j] += p[j];
      if (exact || converged) { status = NLP_OK; break; }
      continue;
    }
    // ---- Armijo backtracking on F (the segment [v, v + p] is feasible) --------------------------------
    double slope = 0.0;
    for (int j = 0; j < N; ++j) slope = fma(g[j], p[j], slope);
    double alpha = 1.0, Ft = F0;
    bool accepted = false;
    for (int k = 0; k < NLP_LS_TRIES; ++k, alpha *= 0.5) {
      for (int j = 0; j < N; ++j) vt[j] = fma(alpha, p[j], v[j]);
      Ft = S::eval_nlp_f(d.P, vt);
      // (a change of F within its rounding is no increase: near the solution F cannot resolve the decrease
      // of a Newton step any more, and refusing it would stall the iteration short of the tolerance)
      if (Ft <= F0 + NLP_ARMIJO_C1 * alpha * slope || Ft - F0 <= NLP_F_FLOOR * fabs(F0) + NLP_F_ABS) {
        accepted = true;
        break;
      }
    }
    if (!accepted) { status = NLP_STALLED; break; }
    for (int j = 0; j < N; ++j) v[j] = vt[j];
    // rounding floor: a small step that no longer changes F beyond rounding ends the iteration as well (the
    // subproblem's own accuracy keeps |p| from reaching tol on ill-conditioned instances)
    if (fabs(F0 - Ft) <= NLP_F_FLOOR * fabs(F0) + NLP_F_ABS &&
        nlp_norm_inf<N>(p) <= NLP_FLOOR_STEP * S::NLP_TOL * (1.0 + nlp_norm_inf<N>(v))) {
      status = NLP_OK;
      break;
    }
  }
  if (status == NLP_OK) {
    for (int j = 0; j < N; ++j) status = finite_bits(v[j]) ? status : NLP_INVALID;
  }
  return status;
}

// Load the inputs of instance i (only the rows the generated program reads: S::NLP_READ_*); false when
// one of them is NaN / inf.
template <class S>
__device__ __forceinline__ bool nlp_load(long long ld, long long i, const double* __restrict__ t, int t_stride,
                                         const double* __restrict__ q, const double* __restrict__ x,
                                         const double* __restrict__ y, double& tv, double (&qv)[S::NQ > 0 ? S::NQ : 1],
                                         double (&xv)[S::NX > 0 ? S::NX : 1], double (&yv)[S::NY > 0 ? S::NY : 1]) {
  tv = S::NLP_READ_T ? t[(long long)t_stride * i] : 0.0;
  bool ok = finite_bits(tv);
  for (int j = 0; j < S::NQ; ++j) {
    qv[j] = row_read(S::NLP_READ_Q, j) ? q[(long long)j * ld + i] : 0.0;
    ok = ok && finite_bits(qv[j]);
  }
  for (int j = 0; j < S::NX; ++j) {
    xv[j] = row_read(S::NLP_READ_X, j) ? x[(long long)j * ld + i] : 0.0;
    ok = ok && finite_bits(xv[j]);
  }
  for (int j = 0; j < S::NY; ++j) {
    yv[j] = row_read(S::NLP_READ_Y, j) ? y[(long long)j * ld + i] : 0.0;
    ok = ok && finite_bits(yv[j]);
  }
  return ok;
}

// Controller step, SoA in / SoA out (layout of qp_step): sol[j*ld + i]; x0 (may be NULL) = start point;
// status, iters (may be NULL); active[i] / active[ld + i] = upper / lower masks (may be NULL).
template <class S>
__device__ __forceinline__ void nlp_step(long long N, long long ld, const double* __restrict__ t, int t_stride,
                                         const double* __restrict__ q, const double* __restrict__ x,
                                         const double* __restrict__ y, const double* __restrict__ x0,
                                         double* __restrict__ sol, int* __restrict__ status, int* __restrict__ iters,
                                         unsigned* __restrict__ active, int max_iter) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    double tv, qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
    const bool data_ok = nlp_load<S>(ld, i, t, t_stride, q, x, y, tv, qv, xv, yv);
    double v[S::NN];
    for (int j = 0; j < S::NN; ++j) v[j] = x0 != nullptr ? x0[(long long)j * ld + i] : 0.0;
    unsigned mu = 0u, ml = 0u;
    int it = 0, st = NLP_INVALID;
    if (data_ok) {
      NlpData<S> d;
      S::eval_nlp_pre(tv, qv, xv, yv, d);
      st = nlp_solve<S>(d, v, &mu, &ml, &it, max_iter);
    }
    if (st == NLP_INVALID) mu = ml = 0u;
    for (int j = 0; j < S::NN; ++j) sol[(long long)j * ld + i] = v[j];
    if (status != nullptr) status[i] = st;
    if (iters != nullptr) iters[i] = it;
    if (active != nullptr) {
      active[i] = mu;
      active[ld + i] = ml;
    }
  }
}

// One step of the closed-loop rollouts (nlp_rollout and the tangent rollouts of clik_jvp.cuh): the SQP
// iteration at (tv, qv, xv, yv) from v, the previous step's solution, which it replaces; (mu, ml) = the last
// subproblem's working set.  Returns the status.
template <class S>
__device__ __forceinline__ int nlp_rollout_solve(double tv, const double (&qv)[S::NQ > 0 ? S::NQ : 1],
                                                 const double (&xv)[S::NX > 0 ? S::NX : 1],
                                                 const double (&yv)[S::NY > 0 ? S::NY : 1], double (&v)[S::NN],
                                                 unsigned& mu, unsigned& ml, int max_iter) {
  NlpData<S> d;
  S::eval_nlp_pre(tv, qv, xv, yv, d);
  int it;
  return nlp_solve<S>(d, v, &mu, &ml, &it, max_iter);
}

// Applies an NLP rollout step: an unsolved one applies zero velocity, is counted in failed and the next step
// starts from zero; xs = v with the robot / virtual parts clipped.
template <class S>
__device__ __forceinline__ void nlp_rollout_advance(int st, double (&v)[S::NN], double (&xs)[S::NN],
                                                    double (&qv)[S::NQ > 0 ? S::NQ : 1],
                                                    double (&xv)[S::NX > 0 ? S::NX : 1], double vmax_q,
                                                    double vmax_x, double dt, int& failed) {
  if (st != NLP_OK) {
    ++failed;
    for (int j = 0; j < S::NN; ++j) v[j] = 0.0;
  }
  for (int j = 0; j < S::NN; ++j) xs[j] = v[j];
  rollout_euler<S>(xs, qv, xv, vmax_q, vmax_x, dt);
}

// Closed-loop rollout (the loop of qp_rollout): each step starts from the previous step's solution,
// v = clip(sol[:n], +-max_speed); q += v_rob*dt; x += v_virt*dt.  A step that is not solved applies zero
// velocity, is counted in n_failed and the next step starts from zero.  sol_last: the last step's
// solution with the robot / virtual parts clipped.
template <class S>
__device__ __forceinline__ void nlp_rollout(long long N, long long ld, int steps, double dt, const double* __restrict__ t0,
                                            int t_stride, double* __restrict__ q, double* __restrict__ x,
                                            const double* __restrict__ y, double vmax_q, double vmax_x,
                                            double* __restrict__ sol_last, int* __restrict__ n_failed, int max_iter) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    double qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
    const double t0v = t0[(long long)t_stride * i];
    for (int j = 0; j < S::NQ; ++j) qv[j] = q[(long long)j * ld + i];
    for (int j = 0; j < S::NX; ++j) xv[j] = x[(long long)j * ld + i];
    for (int j = 0; j < S::NY; ++j) yv[j] = y[(long long)j * ld + i];
    double v[S::NN], xs[S::NN];
    for (int j = 0; j < S::NN; ++j) v[j] = 0.0;
    int failed = 0;
    for (int k = 0; k < steps; ++k) {
      const double tv = __dadd_rn(t0v, __dmul_rn(dt, (double)k));
      unsigned mu, ml;
      const int st = nlp_rollout_solve<S>(tv, qv, xv, yv, v, mu, ml, max_iter);
      nlp_rollout_advance<S>(st, v, xs, qv, xv, vmax_q, vmax_x, dt, failed);
    }
    for (int j = 0; j < S::NQ; ++j) q[(long long)j * ld + i] = qv[j];
    for (int j = 0; j < S::NX; ++j) x[(long long)j * ld + i] = xv[j];
    if (sol_last != nullptr)
      for (int j = 0; j < S::NN; ++j) sol_last[(long long)j * ld + i] = (steps > 0) ? xs[j] : 0.0;
    if (n_failed != nullptr) n_failed[i] = failed;
  }
}

}  // namespace clik
