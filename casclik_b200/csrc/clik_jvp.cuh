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
  __device__ __forceinline__ bool factor(long long ld, long long i, const double* __restrict__ t, int t_stride,
                                         const double* __restrict__ q, const double* __restrict__ x,
                                         const double* __restrict__ y, const double* __restrict__ sol,
                                         const int* __restrict__ status, const unsigned* __restrict__ active) {
    if (status[i] != QP_OK) return false;
    duals_load<S, S::JVP_READ_T, S::JVP_READ_Q, S::JVP_READ_X, S::JVP_READ_Y>(ld, i, t, t_stride, q, x, y, tv, qv, xv,
                                                                              yv);
    S::eval_qp(tv, qv, xv, yv, d);
    up = active[i];
    lo = active[ld + i];
    if (!working_set_rows<NN, M>(up, lo, W, k, lam)) return false;
    for (int j = 0; j < NN; ++j) s[j] = 1.0 / sqrt(d.h[j]);
    for (int a = 0; a < k; ++a)
      for (int j = 0; j < NN; ++j) Q[a * NN + j] = s[j] * d.A[W[a] * NN + j];
    if (!working_set_qr<NN>(k, Q, R)) return false;
    double sg[NN];
    for (int j = 0; j < NN; ++j) {
      xs[j] = sol[(long long)j * ld + i];
      sg[j] = s[j] * (d.h[j] * xs[j]);
    }
    working_set_solve<NN>(k, W, Q, R, sg, lam);
    return true;
  }
  // x_dot from rho1 (stride c) and rho2
  __device__ __forceinline__ void solve(const double* r1, const double* r2u, const double* r2l, int c,
                                        double* xd) const {
    double z[NN];
    for (int j = 0; j < NN; ++j) z[j] = s[j] * -r1[j * c];
    jvp_face_solve<NN>(k, W, Q, R, up, r2u, r2l, c, z);
    for (int j = 0; j < NN; ++j) xd[j] = s[j] * z[j];
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
  __device__ __forceinline__ bool factor(long long ld, long long i, const double* __restrict__ t, int t_stride,
                                         const double* __restrict__ q, const double* __restrict__ x,
                                         const double* __restrict__ y, const double* __restrict__ sol,
                                         const int* __restrict__ status, const unsigned* __restrict__ active) {
    if (status[i] != 0) return false;
    duals_load<S, S::JVP_READ_T, S::JVP_READ_Q, S::JVP_READ_X, S::JVP_READ_Y>(ld, i, t, t_stride, q, x, y, tv, qv, xv,
                                                                              yv);
    NlpData<typename S::Base> d;
    S::eval_nlp_pre(tv, qv, xv, yv, d);
    up = active[i];
    lo = active[ld + i];
    double g[NN], H[NH], one[NN];
    for (int j = 0; j < NN; ++j) {
      xs[j] = sol[(long long)j * ld + i];
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
      nlp_lsolve<NN>(L, &Q[a * NN]);
    }
    return working_set_qr<NN>(k, Q, R);
  }
  __device__ __forceinline__ void solve(const double* r1, const double* r2u, const double* r2l, int c,
                                        double* xd) const {
    for (int j = 0; j < NN; ++j) xd[j] = -r1[j * c];
    nlp_lsolve<NN>(L, xd);
    jvp_face_solve<NN>(k, W, Q, R, up, r2u, r2l, c, xd);
    nlp_ltsolve<NN>(L, xd);
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

}  // namespace clik
