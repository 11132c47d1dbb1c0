// clik_jvp.cuh — forward-mode derivative (Jacobian-vector product) of the QP and NLP controller steps, and the
// full step Jacobian, one instance per thread, fp64, sm_100a.
//
// theta = (t, q, x_virtual, y) of one instance; its step returned x* and the working set W (the two masks of
// `active`; an upper bit selects ub, a lower bit lb, an equality row has both bits and uses ub).  For a tangent
// theta_dot, with x* and lam held fixed,
//
//     rho1   = d_theta (g(x*, theta) + A(theta)' lam) . theta_dot          QP: g = H x,  NLP: g = grad F(x)
//     rho2_r = d_theta (A_r(theta) x* - b_r(theta)) . theta_dot,  r in W
//
// and the face problem of W gives x_dot = (d x*/d theta) theta_dot from
//
//     [[M, A_W'], [A_W, 0]] [x_dot; lam_dot_W] = -[rho1; rho2_W]          M = H (QP), grad^2 F(x*) (NLP).
//
// K is symmetric, so this is the exact adjoint of clik_vjp.cuh: <xb, x_dot> = <theta_bar, theta_dot>.  Where a
// row of W has lam = 0 it is the one-sided derivative that keeps W.
//
// Solve, on the VJP's factorisation B = D^1/2 A_W' = Q R (QP: D = H^-1; NLP: grad^2 F(x*) = L L' unshifted and
// B = L^-1 A_W'): with z = D^-1/2 x_dot (NLP: L' x_dot) and c = -D^1/2 rho1 (NLP: -L^-1 rho1), the system reads
// z + Q R lam_dot = c, R' Q' z = -rho2_W, so w = -R^-T rho2_W and z = (I - Q Q') c + Q w.
// lam is the multipliers routine's own output (same operations in the same order).  Rules, as the VJP's: an
// all-zero tangent gives x_dot = 0 exactly (whatever the status); otherwise x_dot is NaN when the status is not
// 0, when A_W is rank-deficient (the tests of clik_duals.cuh) or, for the NLP, when a Cholesky pivot of
// grad^2 F(x*) is at or below 1e-12 max(1, max_j |H_jj|).  The Jacobian follows the same rules column by column:
// an unsolved or rejected instance gets a block of NaN, and a solved one exact zeros in the columns of theta
// entries the program does not read.
//
// The generated skill provides (codegen/emit.py, emit_skill(..., jvp=True)) S::eval_jvp — rho1 and both forms of
// rho2 (r2u: b = ub, r2l: b = lb) for one tangent — S::eval_jac — the same for every column of theta, entry
// (row, c) at [row * NT + c] — and the read masks JVP_READ_*, on top of S::eval_qp (QP) or S::eval_nlp_pre /
// S::eval_nlp_fgH (NLP) of its base struct S::Base.
#pragma once
#include <cmath>

#include "clik_duals.cuh"

namespace clik {

// w = -R^-T rho2_W by forward substitution (R upper, R[l*N + a] row l column a), then
// z = (I - Q Q') z + Q w: the projection in two passes as working_set_solve, then the range part.  rho2_W[a] is
// r2u[W[a]] for a row with an upper bit, r2l[W[a]] otherwise; `c` is the stride of r2u / r2l.
template <int N>
__device__ __forceinline__ void jvp_face_solve(int k, const int* W, const double* Q, const double* R, unsigned up,
                                               const double* r2u, const double* r2l, int c, double* z) {
  double w[N];
  for (int a = 0; a < k; ++a) {
    const int r = W[a];
    double acc = ((up >> r) & 1u) ? -r2u[r * c] : -r2l[r * c];
    for (int l = 0; l < a; ++l) acc = fma(-R[l * N + a], w[l], acc);
    w[a] = acc / R[a * N + a];
  }
  for (int pass = 0; pass < 2; ++pass) {
    for (int a = 0; a < k; ++a) {
      double dt = 0.0;
      for (int j = 0; j < N; ++j) dt = fma(Q[a * N + j], z[j], dt);
      for (int j = 0; j < N; ++j) z[j] = fma(-dt, Q[a * N + j], z[j]);
    }
  }
  for (int a = 0; a < k; ++a)
    for (int j = 0; j < N; ++j) z[j] = fma(w[a], Q[a * N + j], z[j]);
}

// Instance i's tangent (a NULL array is a zero tangent); true when it is all zeros.
template <class S>
__device__ __forceinline__ bool jvp_tangent(long long ld, long long i, const double* __restrict__ t_dot,
                                            const double* __restrict__ q_dot, const double* __restrict__ x_dot,
                                            const double* __restrict__ y_dot, double& td,
                                            double (&qd)[S::NQ > 0 ? S::NQ : 1], double (&xd)[S::NX > 0 ? S::NX : 1],
                                            double (&yd)[S::NY > 0 ? S::NY : 1]) {
  td = t_dot ? t_dot[i] : 0.0;
  bool zero = td == 0.0;
  for (int j = 0; j < S::NQ; ++j) {
    qd[j] = q_dot ? q_dot[(long long)j * ld + i] : 0.0;
    zero = zero && qd[j] == 0.0;
  }
  for (int j = 0; j < S::NX; ++j) {
    xd[j] = x_dot ? x_dot[(long long)j * ld + i] : 0.0;
    zero = zero && xd[j] == 0.0;
  }
  for (int j = 0; j < S::NY; ++j) {
    yd[j] = y_dot ? y_dot[(long long)j * ld + i] : 0.0;
    zero = zero && yd[j] == 0.0;
  }
  return zero;
}

// The QP face factorisation of instance i (as qp_vjp): rows, s = D^1/2, the QR of D^1/2 A_W' and lam; false when
// the instance is not solved or A_W is rank-deficient.
template <class S>
struct QpFace {
  static constexpr int NN = S::QN, M = S::QM;
  double tv, qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
  QpData<typename S::Base> d;
  unsigned up, lo;
  int W[NN], k;
  double lam[M], Q[NN * NN], R[NN * NN], s[NN], xs[NN];
  // from values in registers: the inputs, the step's solution, status and working set
  __device__ __forceinline__ bool factor(double t_, const double (&q_)[S::NQ > 0 ? S::NQ : 1],
                                         const double (&x_)[S::NX > 0 ? S::NX : 1],
                                         const double (&y_)[S::NY > 0 ? S::NY : 1], const double (&sol_)[NN], int st,
                                         unsigned up_, unsigned lo_) {
    if (st != QP_OK) return false;
    tv = t_;
    for (int j = 0; j < S::NQ; ++j) qv[j] = q_[j];
    for (int j = 0; j < S::NX; ++j) xv[j] = x_[j];
    for (int j = 0; j < S::NY; ++j) yv[j] = y_[j];
    S::eval_qp(tv, qv, xv, yv, d);
    up = up_;
    lo = lo_;
    if (!working_set_rows<NN, M>(up, lo, W, k, lam)) return false;
    for (int j = 0; j < NN; ++j) s[j] = 1.0 / sqrt(d.h[j]);
    for (int a = 0; a < k; ++a)
      for (int j = 0; j < NN; ++j) Q[a * NN + j] = s[j] * d.A[W[a] * NN + j];
    if (!working_set_qr<NN>(k, Q, R)) return false;
    double sg[NN];
    for (int j = 0; j < NN; ++j) {
      xs[j] = sol_[j];
      sg[j] = s[j] * (d.h[j] * xs[j]);
    }
    working_set_solve<NN>(k, W, Q, R, sg, lam);
    return true;
  }
  // of instance i, from global memory
  __device__ __forceinline__ bool factor(long long ld, long long i, const double* __restrict__ t, int t_stride,
                                         const double* __restrict__ q, const double* __restrict__ x,
                                         const double* __restrict__ y, const double* __restrict__ sol,
                                         const int* __restrict__ status, const unsigned* __restrict__ active) {
    if (status[i] != QP_OK) return false;
    duals_load<S, S::JVP_READ_T, S::JVP_READ_Q, S::JVP_READ_X, S::JVP_READ_Y>(ld, i, t, t_stride, q, x, y, tv, qv, xv,
                                                                              yv);
    double sv[NN];
    for (int j = 0; j < NN; ++j) sv[j] = sol[(long long)j * ld + i];
    return factor(tv, qv, xv, yv, sv, QP_OK, active[i], active[ld + i]);
  }
  // x_dot from rho1 (stride c) and rho2
  __device__ __forceinline__ void solve(const double* r1, const double* r2u, const double* r2l, int c,
                                        double* xd) const {
    double z[NN];
    for (int j = 0; j < NN; ++j) z[j] = s[j] * -r1[j * c];
    jvp_face_solve<NN>(k, W, Q, R, up, r2u, r2l, c, z);
    for (int j = 0; j < NN; ++j) xd[j] = s[j] * z[j];
  }
  // the adjoint solve of qp_vjp (the same operations in the same order) for the cotangent xb: K [u; v] = [xb; 0]
  __device__ __forceinline__ void adjoint(const double (&xb)[NN], double (&u)[NN], double (&v)[M]) const {
    for (int r = 0; r < M; ++r) v[r] = 0.0;
    double sg[NN];
    for (int j = 0; j < NN; ++j) sg[j] = s[j] * -xb[j];
    working_set_solve<NN>(k, W, Q, R, sg, v);
    for (int j = 0; j < NN; ++j) {
      double acc = xb[j];
      for (int a = 0; a < k; ++a) acc = fma(-d.A[W[a] * NN + j], v[W[a]], acc);
      u[j] = acc / d.h[j];
    }
  }
};

// The NLP face factorisation of instance i (as nlp_vjp): lam, grad^2 F(x*) = L L' and the QR of L^-1 A_W'.
template <class S>
struct NlpFace {
  static constexpr int NN = S::NN, M = S::NM, NH = S::NN * (S::NN + 1) / 2;
  double tv, qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
  unsigned up, lo;
  int W[NN], k;
  double lam[M], Q[NN * NN], R[NN * NN], L[NH], xs[NN];
  __device__ __forceinline__ bool factor(double t_, const double (&q_)[S::NQ > 0 ? S::NQ : 1],
                                         const double (&x_)[S::NX > 0 ? S::NX : 1],
                                         const double (&y_)[S::NY > 0 ? S::NY : 1], const double (&sol_)[NN], int st,
                                         unsigned up_, unsigned lo_, double* aw = nullptr) {
    if (st != 0) return false;
    tv = t_;
    for (int j = 0; j < S::NQ; ++j) qv[j] = q_[j];
    for (int j = 0; j < S::NX; ++j) xv[j] = x_[j];
    for (int j = 0; j < S::NY; ++j) yv[j] = y_[j];
    NlpData<typename S::Base> d;
    S::eval_nlp_pre(tv, qv, xv, yv, d);
    up = up_;
    lo = lo_;
    double g[NN], H[NH], one[NN];
    for (int j = 0; j < NN; ++j) {
      xs[j] = sol_[j];
      one[j] = 1.0;
    }
    S::eval_nlp_fgH(d.P, xs, g, H);
    if (!working_set_multipliers<NN, M>(d.A, one, g, up, lo, lam)) return false;
    double hmax = 1.0;   // the step's pivot threshold, as nlp_vjp
    for (int j = 0; j < NN; ++j) hmax = fmax(hmax, fabs(H[j * (j + 1) / 2 + j]));
    if (!nlp_cholesky<NN>(H, 0.0, 1e-12 * hmax, L)) return false;
    double v[M];
    if (!working_set_rows<NN, M>(up, lo, W, k, v)) return false;
    for (int a = 0; a < k; ++a) {
      for (int j = 0; j < NN; ++j) Q[a * NN + j] = d.A[W[a] * NN + j];
      if (aw != nullptr)   // the rows of A_W, for NlpAdjointFace
        for (int j = 0; j < NN; ++j) aw[a * NN + j] = Q[a * NN + j];
      nlp_lsolve<NN>(L, &Q[a * NN]);
    }
    return working_set_qr<NN>(k, Q, R);
  }
  __device__ __forceinline__ bool factor(long long ld, long long i, const double* __restrict__ t, int t_stride,
                                         const double* __restrict__ q, const double* __restrict__ x,
                                         const double* __restrict__ y, const double* __restrict__ sol,
                                         const int* __restrict__ status, const unsigned* __restrict__ active) {
    if (status[i] != 0) return false;
    duals_load<S, S::JVP_READ_T, S::JVP_READ_Q, S::JVP_READ_X, S::JVP_READ_Y>(ld, i, t, t_stride, q, x, y, tv, qv, xv,
                                                                              yv);
    double sv[NN];
    for (int j = 0; j < NN; ++j) sv[j] = sol[(long long)j * ld + i];
    return factor(tv, qv, xv, yv, sv, 0, active[i], active[ld + i]);
  }
  __device__ __forceinline__ void solve(const double* r1, const double* r2u, const double* r2l, int c,
                                        double* xd) const {
    for (int j = 0; j < NN; ++j) xd[j] = -r1[j * c];
    nlp_lsolve<NN>(L, xd);
    jvp_face_solve<NN>(k, W, Q, R, up, r2u, r2l, c, xd);
    nlp_ltsolve<NN>(L, xd);
  }
};

// NlpFace that also keeps the rows of A_W, for the adjoint solve of nlp_vjp (the forward-mode kernels do not need
// them and keep the plain NlpFace).
template <class S>
struct NlpAdjointFace : NlpFace<S> {
  using Base = NlpFace<S>;
  static constexpr int NN = Base::NN, M = Base::M;
  double AW[NN * NN];
  __device__ __forceinline__ bool factor(double t_, const double (&q_)[S::NQ > 0 ? S::NQ : 1],
                                         const double (&x_)[S::NX > 0 ? S::NX : 1],
                                         const double (&y_)[S::NY > 0 ? S::NY : 1], const double (&sol_)[NN], int st,
                                         unsigned up_, unsigned lo_) {
    return Base::factor(t_, q_, x_, y_, sol_, st, up_, lo_, AW);
  }
  // the adjoint solve of nlp_vjp (the same operations in the same order): u = L^-T L^-1 (xb - A_W' v)
  __device__ __forceinline__ void adjoint(const double (&xb)[NN], double (&u)[NN], double (&v)[M]) const {
    for (int r = 0; r < M; ++r) v[r] = 0.0;
    double sg[NN];
    for (int j = 0; j < NN; ++j) sg[j] = -xb[j];
    nlp_lsolve<NN>(this->L, sg);
    working_set_solve<NN>(this->k, this->W, this->Q, this->R, sg, v);
    for (int j = 0; j < NN; ++j) {
      double acc = xb[j];
      for (int a = 0; a < this->k; ++a) acc = fma(-AW[a * NN + j], v[this->W[a]], acc);
      u[j] = acc;
    }
    nlp_lsolve<NN>(this->L, u);
    nlp_ltsolve<NN>(this->L, u);
  }
};

// JVP of a step's output (SoA, rows ld apart): sol_dot[j*ld + i].  F: QpFace<S> or NlpFace<S>.
template <class S, class F>
__device__ __forceinline__ void step_jvp(long long N, long long ld, const double* __restrict__ t, int t_stride,
                                         const double* __restrict__ q, const double* __restrict__ x,
                                         const double* __restrict__ y, const double* __restrict__ sol,
                                         const int* __restrict__ status, const unsigned* __restrict__ active,
                                         const double* __restrict__ t_dot, const double* __restrict__ q_dot,
                                         const double* __restrict__ x_dot, const double* __restrict__ y_dot,
                                         double* __restrict__ sol_dot) {
  constexpr int NN = F::NN, M = F::M;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    double out[NN];
    for (int j = 0; j < NN; ++j) out[j] = 0.0;
    double td, qd[S::NQ > 0 ? S::NQ : 1], xd[S::NX > 0 ? S::NX : 1], yd[S::NY > 0 ? S::NY : 1];
    if (!jvp_tangent<S>(ld, i, t_dot, q_dot, x_dot, y_dot, td, qd, xd, yd)) {
      F f;
      if (f.factor(ld, i, t, t_stride, q, x, y, sol, status, active)) {
        double r1[NN], r2u[M], r2l[M];
        S::eval_jvp(f.tv, f.qv, f.xv, f.yv, f.xs, f.lam, td, qd, xd, yd, r1, r2u, r2l);
        f.solve(r1, r2u, r2l, 1, out);
      } else {
        for (int j = 0; j < NN; ++j) out[j] = NAN;
      }
    }
    for (int j = 0; j < NN; ++j) sol_dot[(long long)j * ld + i] = out[j];
  }
}

// Jacobian of a step's output: entry (j, c) of instance i at jac[(j*NT + c)*ld + i], theta ordered (t, q, x, y);
// one factorisation, NT right-hand sides.
template <class S, class F>
__device__ __forceinline__ void step_jacobian(long long N, long long ld, const double* __restrict__ t, int t_stride,
                                              const double* __restrict__ q, const double* __restrict__ x,
                                              const double* __restrict__ y, const double* __restrict__ sol,
                                              const int* __restrict__ status, const unsigned* __restrict__ active,
                                              double* __restrict__ jac) {
  constexpr int NN = F::NN, M = F::M, NT = 1 + S::NQ + S::NX + S::NY;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    F f;
    if (f.factor(ld, i, t, t_stride, q, x, y, sol, status, active)) {
      double r1[NN * NT], r2u[M * NT], r2l[M * NT];
      S::eval_jac(f.tv, f.qv, f.xv, f.yv, f.xs, f.lam, r1, r2u, r2l);
      for (int c = 0; c < NT; ++c) {
        double col[NN];
        f.solve(&r1[c], &r2u[c], &r2l[c], NT, col);
        for (int j = 0; j < NN; ++j) jac[((long long)j * NT + c) * ld + i] = col[j];
      }
    } else {
      for (int j = 0; j < NN * NT; ++j) jac[(long long)j * ld + i] = NAN;
    }
  }
}

template <class S>
__device__ __forceinline__ void qp_jvp(long long N, long long ld, const double* t, int t_stride, const double* q,
                                       const double* x, const double* y, const double* sol, const int* status,
                                       const unsigned* active, const double* t_dot, const double* q_dot,
                                       const double* x_dot, const double* y_dot, double* sol_dot) {
  step_jvp<S, QpFace<S>>(N, ld, t, t_stride, q, x, y, sol, status, active, t_dot, q_dot, x_dot, y_dot, sol_dot);
}

template <class S>
__device__ __forceinline__ void nlp_jvp(long long N, long long ld, const double* t, int t_stride, const double* q,
                                        const double* x, const double* y, const double* sol, const int* status,
                                        const unsigned* active, const double* t_dot, const double* q_dot,
                                        const double* x_dot, const double* y_dot, double* sol_dot) {
  step_jvp<S, NlpFace<S>>(N, ld, t, t_stride, q, x, y, sol, status, active, t_dot, q_dot, x_dot, y_dot, sol_dot);
}

template <class S>
__device__ __forceinline__ void qp_jacobian(long long N, long long ld, const double* t, int t_stride, const double* q,
                                            const double* x, const double* y, const double* sol, const int* status,
                                            const unsigned* active, double* jac) {
  step_jacobian<S, QpFace<S>>(N, ld, t, t_stride, q, x, y, sol, status, active, jac);
}

template <class S>
__device__ __forceinline__ void nlp_jacobian(long long N, long long ld, const double* t, int t_stride, const double* q,
                                             const double* x, const double* y, const double* sol, const int* status,
                                             const unsigned* active, double* jac) {
  step_jacobian<S, NlpFace<S>>(N, ld, t, t_stride, q, x, y, sol, status, active, jac);
}

// ---- forward-mode derivative of the closed-loop rollouts ------------------------------------------------------
//
// The rollout of qp_rollout / nlp_rollout (the same step helpers, hence the same primal bits) with the tangent of
// the state carried next to it.  p = (t0, q0, x0, y); at step k theta_k = (t0 + k dt, q_k, x_k, y), sol_k the
// step's unclipped solution and active_k its working set.  Per step:
//   s_dot_k = the step JVP above at (theta_k, sol_k, status_k, active_k) along theta_dot_k = (t0_dot, q_dot_k,
//             x_dot_k, y_dot): exactly 0 for an all-zero theta_dot_k, NaN under the step JVP's rules; once NaN, the
//             instance's tangent outputs are NaN from then on;
//   v_dot_j  = s_dot_j where |sol_j| < vmax (vmax_q robot part, vmax_x virtual part), 0 where the clip holds (at
//             the bound too); slack entries are not clipped;
//   q_dot_{k+1} = q_dot_k + dt v_dot_q,  x_dot_{k+1} = x_dot_k + dt v_dot_x  (the rounding of the primal update).
// The face of step k is factored from registers before the solution is clipped into the next step's start.
// The Jacobian rollout carries P = d(q_k, x_k)/dp (NS x NT) instead: one eval_jac and one factorisation per step,
// rho contracted with d theta_k / dp = [e_0; P; 0 I], then NT face solves.

// The primal of one instance's QP rollout: qp_rollout_solve / qp_rollout_advance, as qp_rollout.  P = the step
// skill (the struct qp_rollout is instantiated on), S = its JVP struct.
template <class S, class P>
struct QpRolloutState {
  using Face = QpFace<S>;
  static constexpr int NN = S::QN;
  double xs[NN];             // the step's unclipped solution after solve(), clipped after advance()
  unsigned mu = 0u, ml = 0u;  // working set of the previous step = warm start of the next
  int st = QP_OK;
  __device__ __forceinline__ QpRolloutState() {
    for (int j = 0; j < NN; ++j) xs[j] = 0.0;
  }
  __device__ __forceinline__ void solve(double tv, const double (&qv)[S::NQ > 0 ? S::NQ : 1],
                                        const double (&xv)[S::NX > 0 ? S::NX : 1],
                                        const double (&yv)[S::NY > 0 ? S::NY : 1], int max_iter) {
    st = qp_rollout_solve<P>(tv, qv, xv, yv, xs, mu, ml, max_iter);
  }
  __device__ __forceinline__ const double (&sol() const)[NN] { return xs; }
  __device__ __forceinline__ void advance(double (&qv)[S::NQ > 0 ? S::NQ : 1], double (&xv)[S::NX > 0 ? S::NX : 1],
                                          double vmax_q, double vmax_x, double dt, int& failed) {
    qp_rollout_advance<P>(st, xs, qv, xv, vmax_q, vmax_x, dt, failed);
  }
  __device__ __forceinline__ double last(int j, int) const { return xs[j]; }
};

// The primal of one instance's NLP rollout: nlp_rollout_solve / nlp_rollout_advance, as nlp_rollout.
template <class S, class P>
struct NlpRolloutState {
  using Face = NlpFace<S>;
  static constexpr int NN = S::NN;
  double v[NN], xs[NN];      // v: the step's solution and the next step's start; xs: v clipped
  unsigned mu = 0u, ml = 0u;
  int st = 0;
  __device__ __forceinline__ NlpRolloutState() {
    for (int j = 0; j < NN; ++j) v[j] = 0.0;
  }
  __device__ __forceinline__ void solve(double tv, const double (&qv)[S::NQ > 0 ? S::NQ : 1],
                                        const double (&xv)[S::NX > 0 ? S::NX : 1],
                                        const double (&yv)[S::NY > 0 ? S::NY : 1], int max_iter) {
    st = nlp_rollout_solve<P>(tv, qv, xv, yv, v, mu, ml, max_iter);
  }
  __device__ __forceinline__ const double (&sol() const)[NN] { return v; }
  __device__ __forceinline__ void advance(double (&qv)[S::NQ > 0 ? S::NQ : 1], double (&xv)[S::NX > 0 ? S::NX : 1],
                                          double vmax_q, double vmax_x, double dt, int& failed) {
    nlp_rollout_advance<P>(st, v, xs, qv, xv, vmax_q, vmax_x, dt, failed);
  }
  __device__ __forceinline__ double last(int j, int steps) const { return steps > 0 ? xs[j] : 0.0; }
};

// The clip mask of a step's tangent (entries j < NQ + NX of s_dot) and the Euler update of the state tangent.
template <class S>
__device__ __forceinline__ double clip_tangent(int j, double sol_j, double s_dot_j, double vmax_q, double vmax_x) {
  return fabs(sol_j) < (j < S::NQ ? vmax_q : vmax_x) ? s_dot_j : 0.0;
}

// Tangent rollout (JAC false: q_dot_out, x_dot_out, sol_dot) or Jacobian rollout (JAC true: jac, entry (s, c) of
// instance i at jac[(s*NT + c)*ld + i], s over (q, x), c over p), with the primal outputs of the rollout kernels.
// R: QpRolloutState<S, P> or NlpRolloutState<S, P>.
template <class S, class R, bool JAC>
__device__ __forceinline__ void rollout_tangent(long long N, long long ld, int steps, double dt,
                                                const double* __restrict__ t0, int t_stride, double* __restrict__ q,
                                                double* __restrict__ x, const double* __restrict__ y, double vmax_q,
                                                double vmax_x, double* __restrict__ sol_last,
                                                int* __restrict__ n_failed, int max_iter,
                                                const double* __restrict__ t_dot, const double* __restrict__ q_dot,
                                                const double* __restrict__ x_dot, const double* __restrict__ y_dot,
                                                double* __restrict__ q_dot_out, double* __restrict__ x_dot_out,
                                                double* __restrict__ sol_dot, double* __restrict__ jac) {
  using F = typename R::Face;
  constexpr int NN = F::NN, M = F::M, NQ = S::NQ, NX = S::NX, NY = S::NY, NS = NQ + NX, NT = 1 + NS + NY;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    double qv[NQ > 0 ? NQ : 1], xv[NX > 0 ? NX : 1], yv[NY > 0 ? NY : 1];
    const double t0v = t0[(long long)t_stride * i];
    for (int j = 0; j < NQ; ++j) qv[j] = q[(long long)j * ld + i];
    for (int j = 0; j < NX; ++j) xv[j] = x[(long long)j * ld + i];
    for (int j = 0; j < NY; ++j) yv[j] = y[(long long)j * ld + i];
    double td, qd[NQ > 0 ? NQ : 1], xd[NX > 0 ? NX : 1], yd[NY > 0 ? NY : 1];   // JVP: the state's tangent
    double sd[NN];                                                              // JVP: s_dot of the last step
    double Pm[JAC ? NS * NT : 1];                                               // Jacobian: d(q, x)/dp
    if constexpr (JAC) {
      for (int a = 0; a < NS * NT; ++a) Pm[a] = 0.0;
      for (int a = 0; a < NS; ++a) Pm[a * NT + 1 + a] = 1.0;
    } else {
      jvp_tangent<S>(ld, i, t_dot, q_dot, x_dot, y_dot, td, qd, xd, yd);
      for (int j = 0; j < NN; ++j) sd[j] = 0.0;
    }
    bool dead = false;   // a NaN derivative: every later one is NaN
    int failed = 0;
    R r;
    for (int k = 0; k < steps; ++k) {
      const double tv = __dadd_rn(t0v, __dmul_rn(dt, (double)k));
      r.solve(tv, qv, xv, yv, max_iter);
      if constexpr (JAC) {
        if (!dead) {
          F f;
          if (f.factor(tv, qv, xv, yv, r.sol(), r.st, r.mu, r.ml)) {
            double r1[NN * NT], r2u[M * NT], r2l[M * NT];
            S::eval_jac(f.tv, f.qv, f.xv, f.yv, f.xs, f.lam, r1, r2u, r2l);
            // d rho / dp = d rho / d theta_k . d theta_k / dp, row by row in place
            auto chain = [&](double* row) {
              double out[NT];
              for (int c = 0; c < NT; ++c) {
                double acc = (c == 0 || c > NS) ? row[c] : 0.0;
                for (int a = 0; a < NS; ++a) acc = fma(row[1 + a], Pm[a * NT + c], acc);
                out[c] = acc;
              }
              for (int c = 0; c < NT; ++c) row[c] = out[c];
            };
            for (int j = 0; j < NN; ++j) chain(&r1[j * NT]);
            for (int a = 0; a < M; ++a) {
              chain(&r2u[a * NT]);
              chain(&r2l[a * NT]);
            }
            for (int c = 0; c < NT; ++c) {
              double col[NN];
              f.solve(&r1[c], &r2u[c], &r2l[c], NT, col);
              for (int a = 0; a < NS; ++a)
                Pm[a * NT + c] = __dadd_rn(Pm[a * NT + c],
                                           __dmul_rn(clip_tangent<S>(a, r.sol()[a], col[a], vmax_q, vmax_x), dt));
            }
          } else {
            dead = true;
          }
        }
      } else {
        bool zero = td == 0.0;
        for (int j = 0; j < NQ; ++j) zero = zero && qd[j] == 0.0;
        for (int j = 0; j < NX; ++j) zero = zero && xd[j] == 0.0;
        for (int j = 0; j < NY; ++j) zero = zero && yd[j] == 0.0;
        if (zero) {
          for (int j = 0; j < NN; ++j) sd[j] = 0.0;
        } else if (!dead) {
          F f;
          if (f.factor(tv, qv, xv, yv, r.sol(), r.st, r.mu, r.ml)) {
            double r1[NN], r2u[M], r2l[M];
            S::eval_jvp(f.tv, f.qv, f.xv, f.yv, f.xs, f.lam, td, qd, xd, yd, r1, r2u, r2l);
            f.solve(r1, r2u, r2l, 1, sd);
            for (int j = 0; j < NS; ++j) sd[j] = clip_tangent<S>(j, r.sol()[j], sd[j], vmax_q, vmax_x);
            for (int j = 0; j < NQ; ++j) qd[j] = __dadd_rn(qd[j], __dmul_rn(sd[j], dt));
            for (int j = 0; j < NX; ++j) xd[j] = __dadd_rn(xd[j], __dmul_rn(sd[NQ + j], dt));
          } else {
            dead = true;
          }
        }
      }
      r.advance(qv, xv, vmax_q, vmax_x, dt, failed);
    }
    for (int j = 0; j < NQ; ++j) q[(long long)j * ld + i] = qv[j];
    for (int j = 0; j < NX; ++j) x[(long long)j * ld + i] = xv[j];
    if (sol_last != nullptr)
      for (int j = 0; j < NN; ++j) sol_last[(long long)j * ld + i] = r.last(j, steps);
    if (n_failed != nullptr) n_failed[i] = failed;
    if constexpr (JAC) {
      for (int a = 0; a < NS * NT; ++a) jac[(long long)a * ld + i] = dead ? NAN : Pm[a];
    } else {
      for (int j = 0; j < NQ; ++j) q_dot_out[(long long)j * ld + i] = dead ? NAN : qd[j];
      for (int j = 0; j < NX; ++j) x_dot_out[(long long)j * ld + i] = dead ? NAN : xd[j];
      if (sol_dot != nullptr)
        for (int j = 0; j < NN; ++j) sol_dot[(long long)j * ld + i] = dead ? NAN : sd[j];
    }
  }
}

template <class S, class P>
__device__ __forceinline__ void qp_rollout_jvp(long long N, long long ld, int steps, double dt, const double* t0,
                                               int t_stride, double* q, double* x, const double* y, double vmax_q,
                                               double vmax_x, double* sol_last, int* n_failed, int max_iter,
                                               const double* t_dot, const double* q_dot, const double* x_dot,
                                               const double* y_dot, double* q_dot_out, double* x_dot_out,
                                               double* sol_dot) {
  rollout_tangent<S, QpRolloutState<S, P>, false>(N, ld, steps, dt, t0, t_stride, q, x, y, vmax_q, vmax_x, sol_last,
                                                  n_failed, max_iter, t_dot, q_dot, x_dot, y_dot, q_dot_out,
                                                  x_dot_out, sol_dot, nullptr);
}

template <class S, class P>
__device__ __forceinline__ void nlp_rollout_jvp(long long N, long long ld, int steps, double dt, const double* t0,
                                                int t_stride, double* q, double* x, const double* y, double vmax_q,
                                                double vmax_x, double* sol_last, int* n_failed, int max_iter,
                                                const double* t_dot, const double* q_dot, const double* x_dot,
                                                const double* y_dot, double* q_dot_out, double* x_dot_out,
                                                double* sol_dot) {
  rollout_tangent<S, NlpRolloutState<S, P>, false>(N, ld, steps, dt, t0, t_stride, q, x, y, vmax_q, vmax_x, sol_last,
                                                   n_failed, max_iter, t_dot, q_dot, x_dot, y_dot, q_dot_out,
                                                   x_dot_out, sol_dot, nullptr);
}

template <class S, class P>
__device__ __forceinline__ void qp_rollout_jacobian(long long N, long long ld, int steps, double dt, const double* t0,
                                                    int t_stride, double* q, double* x, const double* y,
                                                    double vmax_q, double vmax_x, double* sol_last, int* n_failed,
                                                    int max_iter, double* jac) {
  rollout_tangent<S, QpRolloutState<S, P>, true>(N, ld, steps, dt, t0, t_stride, q, x, y, vmax_q, vmax_x, sol_last,
                                                 n_failed, max_iter, nullptr, nullptr, nullptr, nullptr, nullptr,
                                                 nullptr, nullptr, jac);
}

template <class S, class P>
__device__ __forceinline__ void nlp_rollout_jacobian(long long N, long long ld, int steps, double dt, const double* t0,
                                                     int t_stride, double* q, double* x, const double* y,
                                                     double vmax_q, double vmax_x, double* sol_last, int* n_failed,
                                                     int max_iter, double* jac) {
  rollout_tangent<S, NlpRolloutState<S, P>, true>(N, ld, steps, dt, t0, t_stride, q, x, y, vmax_q, vmax_x, sol_last,
                                                  n_failed, max_iter, nullptr, nullptr, nullptr, nullptr, nullptr,
                                                  nullptr, nullptr, jac);
}

}  // namespace clik
