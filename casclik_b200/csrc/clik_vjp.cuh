// clik_vjp.cuh — reverse-mode derivative (vector-Jacobian product) of the QP and NLP controller steps, one
// instance per thread, fp64, sm_100a.
//
// theta = (t, q, x_virtual, y) of one instance; its step returned x* and the working set W (the two masks of
// `active`).  On W the step solves
//
//     r1 = g(x, theta) + A_W(theta)' lam_W = 0        QP: g = H(theta) x,   NLP: g = grad F(x, theta)
//     r2 = A_W(theta) x - b_W(theta)       = 0        b_r = ub_r (upper bit) or lb_r (lower bit)
//
// with K = d(r1, r2)/d(x, lam) = [[M, A_W'], [A_W, 0]], M = H (QP) or grad^2 F(x*) (NLP).  For a cotangent xb
// the adjoint system K [u; v] = [xb; 0] gives
//
//     theta_bar = -grad_theta Phi,   Phi = u'(g(x*, theta) + A(theta)' lam) + v'(A_W(theta) x* - b_W(theta))
//
// with x*, lam, u, v held fixed: (d x*/d theta)' xb of the face problem of W.  It is the derivative of the step
// where strict complementarity holds; where a row of W has lam = 0 it is the one-sided derivative that keeps W.
//
// Adjoint solve (the least-squares solve of clik_duals.cuh with another right-hand side):
//   QP:  v = argmin |D^1/2 (-xb + A_W' v)|, D = H^-1 (the multipliers' QR, reused), u = D (xb - A_W' v);
//   NLP: grad^2 F(x*) = L L' (no shift), columns L^-1 a_r, pre-scaled gradient -L^-1 xb, u = L^-T L^-1 (xb - A_W' v).
// lam is the multipliers routine's own output.  Rules: an all-zero cotangent column gives theta_bar = 0 exactly
// (whatever the status); otherwise theta_bar is NaN when the status is not 0, when A_W is rank-deficient (the
// tests of clik_duals.cuh) or, for the NLP, when a Cholesky pivot of grad^2 F(x*) is at or below
// 1e-12 max(1, max_j |H_jj|), the step's own threshold (singular or indefinite to working precision).
//
// The generated skill provides (codegen/emit.py, emit_skill(..., vjp=True)) S::eval_vjp — the gradient program
// of Phi over the skill's expression graph — and the read masks VJP_READ_* (rows eval_vjp and the row evaluation
// read), on top of S::eval_qp (QP) or S::eval_nlp_pre / S::eval_nlp_fgH (NLP) of its base struct S::Base.
#pragma once
#include <cmath>

#include "clik_duals.cuh"

namespace clik {

template <class S>
struct VjpOut {
  double t;
  double q[S::NQ > 0 ? S::NQ : 1], x[S::NX > 0 ? S::NX : 1], y[S::NY > 0 ? S::NY : 1];
  __device__ __forceinline__ void fill(double v) {
    t = v;
    for (int j = 0; j < S::NQ; ++j) q[j] = v;
    for (int j = 0; j < S::NX; ++j) x[j] = v;
    for (int j = 0; j < S::NY; ++j) y[j] = v;
  }
  __device__ __forceinline__ void store(long long ld, long long i, double* __restrict__ t_bar,
                                        double* __restrict__ q_bar, double* __restrict__ x_bar,
                                        double* __restrict__ y_bar) const {
    t_bar[i] = t;
    for (int j = 0; j < S::NQ; ++j) q_bar[(long long)j * ld + i] = q[j];
    for (int j = 0; j < S::NX; ++j) x_bar[(long long)j * ld + i] = x[j];
    for (int j = 0; j < S::NY; ++j) y_bar[(long long)j * ld + i] = y[j];
  }
};

// vu / vl: the adjoint v on the rows held at their upper / lower bound (an upper bit selects ub), 0 elsewhere
template <int M>
__device__ __forceinline__ void vjp_split_v(const double* v, unsigned up, unsigned lo, double* vu, double* vl) {
  for (int r = 0; r < M; ++r) {
    const bool u = (up >> r) & 1u, l = (lo >> r) & 1u;
    vu[r] = u ? v[r] : 0.0;
    vl[r] = (l && !u) ? v[r] : 0.0;
  }
}

// Reads instance i's cotangent; true when the column is all zeros.
template <int N>
__device__ __forceinline__ bool vjp_cotangent(long long ld, long long i, const double* __restrict__ sol_bar,
                                              double* xb) {
  bool zero = true;
  for (int j = 0; j < N; ++j) {
    xb[j] = sol_bar[(long long)j * ld + i];
    zero = zero && xb[j] == 0.0;
  }
  return zero;
}

// VJP of clik_qp_step's output (SoA, rows ld apart): t_bar[i], q_bar / x_bar / y_bar[j*ld + i].
template <class S>
__device__ __forceinline__ void qp_vjp(long long N, long long ld, const double* __restrict__ t, int t_stride,
                                       const double* __restrict__ q, const double* __restrict__ x,
                                       const double* __restrict__ y, const double* __restrict__ sol,
                                       const int* __restrict__ status, const unsigned* __restrict__ active,
                                       const double* __restrict__ sol_bar, double* __restrict__ t_bar,
                                       double* __restrict__ q_bar, double* __restrict__ x_bar,
                                       double* __restrict__ y_bar) {
  constexpr int NN = S::QN, M = S::QM;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    VjpOut<S> o;
    o.fill(0.0);
    double xb[NN];
    if (!vjp_cotangent<NN>(ld, i, sol_bar, xb)) {
      bool ok = status[i] == QP_OK;
      if (ok) {
        double tv, qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
        duals_load<S, S::VJP_READ_T, S::VJP_READ_Q, S::VJP_READ_X, S::VJP_READ_Y>(ld, i, t, t_stride, q, x, y, tv, qv,
                                                                                  xv, yv);
        QpData<typename S::Base> d;
        S::eval_qp(tv, qv, xv, yv, d);
        const unsigned up = active[i], lo = active[ld + i];
        int W[NN], k;
        double lam[M], v[M], Q[NN * NN], R[NN * NN], s[NN], xs[NN], sg[NN];
        ok = working_set_rows<NN, M>(up, lo, W, k, lam);
        if (ok) {
          for (int j = 0; j < NN; ++j) s[j] = 1.0 / sqrt(d.h[j]);
          for (int a = 0; a < k; ++a)
            for (int j = 0; j < NN; ++j) Q[a * NN + j] = s[j] * d.A[W[a] * NN + j];
          ok = working_set_qr<NN>(k, Q, R);
        }
        if (ok) {
          // multipliers (as qp_duals: g = H x*), then the adjoint with g = -xb on the same factorisation
          for (int j = 0; j < NN; ++j) {
            xs[j] = sol[(long long)j * ld + i];
            sg[j] = s[j] * (d.h[j] * xs[j]);
          }
          working_set_solve<NN>(k, W, Q, R, sg, lam);
          for (int r = 0; r < M; ++r) v[r] = 0.0;
          for (int j = 0; j < NN; ++j) sg[j] = s[j] * -xb[j];
          working_set_solve<NN>(k, W, Q, R, sg, v);
          double u[NN], vu[M], vl[M];
          for (int j = 0; j < NN; ++j) {
            double acc = xb[j];
            for (int a = 0; a < k; ++a) acc = fma(-d.A[W[a] * NN + j], v[W[a]], acc);
            u[j] = acc / d.h[j];
          }
          vjp_split_v<M>(v, up, lo, vu, vl);
          S::eval_vjp(tv, qv, xv, yv, xs, lam, u, vu, vl, o.t, o.q, o.x, o.y);
        }
      }
      if (!ok) o.fill(NAN);
    }
    o.store(ld, i, t_bar, q_bar, x_bar, y_bar);
  }
}

// VJP of clik_nlp_step's output, as qp_vjp.
template <class S>
__device__ __forceinline__ void nlp_vjp(long long N, long long ld, const double* __restrict__ t, int t_stride,
                                        const double* __restrict__ q, const double* __restrict__ x,
                                        const double* __restrict__ y, const double* __restrict__ sol,
                                        const int* __restrict__ status, const unsigned* __restrict__ active,
                                        const double* __restrict__ sol_bar, double* __restrict__ t_bar,
                                        double* __restrict__ q_bar, double* __restrict__ x_bar,
                                        double* __restrict__ y_bar) {
  constexpr int NN = S::NN, M = S::NM, NH = S::NN * (S::NN + 1) / 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    VjpOut<S> o;
    o.fill(0.0);
    double xb[NN];
    if (!vjp_cotangent<NN>(ld, i, sol_bar, xb)) {
      bool ok = status[i] == 0;
      if (ok) {
        double tv, qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
        duals_load<S, S::VJP_READ_T, S::VJP_READ_Q, S::VJP_READ_X, S::VJP_READ_Y>(ld, i, t, t_stride, q, x, y, tv, qv,
                                                                                  xv, yv);
        NlpData<typename S::Base> d;
        S::eval_nlp_pre(tv, qv, xv, yv, d);
        const unsigned up = active[i], lo = active[ld + i];
        double xs[NN], g[NN], H[NH], L[NH], one[NN], lam[M];
        for (int j = 0; j < NN; ++j) {
          xs[j] = sol[(long long)j * ld + i];
          one[j] = 1.0;
        }
        S::eval_nlp_fgH(d.P, xs, g, H);
        ok = working_set_multipliers<NN, M>(d.A, one, g, up, lo, lam);
        // the step's pivot threshold (clik_nlp.cuh): on a singular Hessian the trailing pivots are rounding noise of
        // either sign, and a positive one would give a finite theta_bar of that noise
        double hmax = 1.0;
        for (int j = 0; j < NN; ++j) hmax = fmax(hmax, fabs(H[j * (j + 1) / 2 + j]));
        if (ok) ok = nlp_cholesky<NN>(H, 0.0, 1e-12 * hmax, L);
        int W[NN], k;
        double v[M], Q[NN * NN], R[NN * NN];
        if (ok) ok = working_set_rows<NN, M>(up, lo, W, k, v);
        if (ok) {
          for (int a = 0; a < k; ++a) {
            for (int j = 0; j < NN; ++j) Q[a * NN + j] = d.A[W[a] * NN + j];
            nlp_lsolve<NN>(L, &Q[a * NN]);
          }
          ok = working_set_qr<NN>(k, Q, R);
        }
        if (ok) {
          double sg[NN], u[NN], vu[M], vl[M];
          for (int j = 0; j < NN; ++j) sg[j] = -xb[j];
          nlp_lsolve<NN>(L, sg);
          working_set_solve<NN>(k, W, Q, R, sg, v);
          for (int j = 0; j < NN; ++j) {
            double acc = xb[j];
            for (int a = 0; a < k; ++a) acc = fma(-d.A[W[a] * NN + j], v[W[a]], acc);
            u[j] = acc;
          }
          nlp_lsolve<NN>(L, u);
          nlp_ltsolve<NN>(L, u);
          vjp_split_v<M>(v, up, lo, vu, vl);
          S::eval_vjp(tv, qv, xv, yv, xs, lam, u, vu, vl, o.t, o.q, o.x, o.y);
        }
      }
      if (!ok) o.fill(NAN);
    }
    o.store(ld, i, t_bar, q_bar, x_bar, y_bar);
  }
}

}  // namespace clik
