// clik_rollout_vjp.cuh — reverse-mode derivative of the QP and NLP closed-loop rollouts: a taped rollout and the
// reverse sweep over its tape, one instance per thread, fp64, sm_100a.
//
// p = (t0, q0, x0, y); the primal is the loop of qp_rollout / nlp_rollout (the same step helpers, hence the same
// bits), t_k = t0 + k dt.  The caller's cotangents are those of q_K, x_K and sol (the clipped last solution).
//
// Tape (rollout_tape), step-major, step k's block in the SoA layout of the step kernels (rows ld apart):
//   q (NQ, ld): q_k, the state at the start of the step     x (NX, ld): x_k
//   sol (NN, ld): the step's unclipped solution             status (ld)     active (2, ld): its working set
// so that step k of the tape is a valid input of the step VJP kernel.
//
// Sweep (rollout_vjp), a_q = q_bar_K, a_x = x_bar_K, for k = K-1 ... 0:
//   s_bar_k = m_k * (dt [a_q; a_x; 0] + [k = K-1] sol_bar)   m_kj = 1 where |sol_kj| < vmax (vmax_q robot part,
//             vmax_x virtual part), 0 where the clip holds (at the bound too); slack entries are not clipped
//   theta_bar_k = the step VJP (clik_vjp.cuh) at (theta_k, sol_k, status_k, active_k) along s_bar_k: exactly 0 for
//             an all-zero s_bar_k (the face is not factored); NaN under the step VJP's rules, and then every
//             cotangent output of the instance is NaN
//   a_q += theta_bar_k.q,  a_x += theta_bar_k.x,  t0_bar += theta_bar_k.t,  y_bar += theta_bar_k.y
// -> q0_bar = a_q, x0_bar = a_x, t0_bar, y_bar: the exact adjoint of the tangent rollout of clik_jvp.cuh.  The
// state cotangent lives in registers; per step the sweep reads the tape and runs one face factorisation
// (QpFace / NlpFace), one adjoint solve and one eval_vjp.
#pragma once
#include <cmath>

#include "clik_jvp.cuh"
#include "clik_vjp.cuh"

namespace clik {

// The rollout of rollout_tangent's primal (q, x, sol_last, n_failed bit-identical to the rollout kernels) writing
// the tape.  R: QpRolloutState<S, P> or NlpRolloutState<S, P>.
template <class S, class R>
__device__ __forceinline__ void rollout_tape(long long N, long long ld, int steps, double dt,
                                             const double* __restrict__ t0, int t_stride, double* __restrict__ q,
                                             double* __restrict__ x, const double* __restrict__ y, double vmax_q,
                                             double vmax_x, double* __restrict__ sol_last, int* __restrict__ n_failed,
                                             int max_iter, double* __restrict__ tape_q, double* __restrict__ tape_x,
                                             double* __restrict__ tape_sol, int* __restrict__ tape_status,
                                             unsigned* __restrict__ tape_active) {
  constexpr int NN = R::NN, NQ = S::NQ, NX = S::NX, NY = S::NY;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    double qv[NQ > 0 ? NQ : 1], xv[NX > 0 ? NX : 1], yv[NY > 0 ? NY : 1];
    const double t0v = t0[(long long)t_stride * i];
    for (int j = 0; j < NQ; ++j) qv[j] = q[(long long)j * ld + i];
    for (int j = 0; j < NX; ++j) xv[j] = x[(long long)j * ld + i];
    for (int j = 0; j < NY; ++j) yv[j] = y[(long long)j * ld + i];
    int failed = 0;
    R r;
    for (int k = 0; k < steps; ++k) {
      for (int j = 0; j < NQ; ++j) tape_q[((long long)k * NQ + j) * ld + i] = qv[j];
      for (int j = 0; j < NX; ++j) tape_x[((long long)k * NX + j) * ld + i] = xv[j];
      const double tv = __dadd_rn(t0v, __dmul_rn(dt, (double)k));
      r.solve(tv, qv, xv, yv, max_iter);
      for (int j = 0; j < NN; ++j) tape_sol[((long long)k * NN + j) * ld + i] = r.sol()[j];
      tape_status[(long long)k * ld + i] = r.st;
      tape_active[(long long)(2 * k) * ld + i] = r.mu;
      tape_active[(long long)(2 * k + 1) * ld + i] = r.ml;
      r.advance(qv, xv, vmax_q, vmax_x, dt, failed);
    }
    for (int j = 0; j < NQ; ++j) q[(long long)j * ld + i] = qv[j];
    for (int j = 0; j < NX; ++j) x[(long long)j * ld + i] = xv[j];
    if (sol_last != nullptr)
      for (int j = 0; j < NN; ++j) sol_last[(long long)j * ld + i] = r.last(j, steps);
    if (n_failed != nullptr) n_failed[i] = failed;
  }
}

// The reverse sweep over a tape of rollout_tape.  F: QpFace<S> or NlpAdjointFace<S>; a NULL cotangent is zero.
template <class S, class F>
__device__ __forceinline__ void rollout_vjp(long long N, long long ld, int steps, double dt,
                                            const double* __restrict__ t0, int t_stride, const double* __restrict__ y,
                                            double vmax_q, double vmax_x, const double* __restrict__ tape_q,
                                            const double* __restrict__ tape_x, const double* __restrict__ tape_sol,
                                            const int* __restrict__ tape_status,
                                            const unsigned* __restrict__ tape_active,
                                            const double* __restrict__ q_bar_K, const double* __restrict__ x_bar_K,
                                            const double* __restrict__ sol_bar, double* __restrict__ t_bar,
                                            double* __restrict__ q_bar, double* __restrict__ x_bar,
                                            double* __restrict__ y_bar) {
  constexpr int NN = F::NN, M = F::M, NQ = S::NQ, NX = S::NX, NY = S::NY, NS = NQ + NX;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    const double t0v = t0[(long long)t_stride * i];
    double yv[NY > 0 ? NY : 1];
    for (int j = 0; j < NY; ++j) yv[j] = y[(long long)j * ld + i];
    VjpOut<S> a;   // a.q, a.x: the state cotangent; a.t, a.y: the accumulated t0_bar and y_bar
    a.fill(0.0);
    for (int j = 0; j < NQ; ++j) a.q[j] = q_bar_K ? q_bar_K[(long long)j * ld + i] : 0.0;
    for (int j = 0; j < NX; ++j) a.x[j] = x_bar_K ? x_bar_K[(long long)j * ld + i] : 0.0;
    bool dead = false;
    for (int k = steps - 1; k >= 0; --k) {
      double sk[NN], xb[NN];
      bool zero = true;
      for (int j = 0; j < NN; ++j) {
        sk[j] = tape_sol[((long long)k * NN + j) * ld + i];
        double c = j < NQ ? __dmul_rn(dt, a.q[j]) : j < NS ? __dmul_rn(dt, a.x[j - NQ]) : 0.0;
        if (k == steps - 1 && sol_bar != nullptr) c = __dadd_rn(c, sol_bar[(long long)j * ld + i]);
        xb[j] = j < NS ? clip_tangent<S>(j, sk[j], c, vmax_q, vmax_x) : c;
        zero = zero && xb[j] == 0.0;
      }
      if (zero) continue;
      double qk[NQ > 0 ? NQ : 1], xk[NX > 0 ? NX : 1];
      for (int j = 0; j < NQ; ++j) qk[j] = tape_q[((long long)k * NQ + j) * ld + i];
      for (int j = 0; j < NX; ++j) xk[j] = tape_x[((long long)k * NX + j) * ld + i];
      const double tv = __dadd_rn(t0v, __dmul_rn(dt, (double)k));
      F f;
      if (!f.factor(tv, qk, xk, yv, sk, tape_status[(long long)k * ld + i], tape_active[(long long)(2 * k) * ld + i],
                    tape_active[(long long)(2 * k + 1) * ld + i])) {
        dead = true;
        break;
      }
      double u[NN], v[M], vu[M], vl[M];
      f.adjoint(xb, u, v);
      vjp_split_v<M>(v, f.up, f.lo, vu, vl);
      VjpOut<S> o;
      o.fill(0.0);
      S::eval_vjp(f.tv, f.qv, f.xv, f.yv, f.xs, f.lam, u, vu, vl, o.t, o.q, o.x, o.y);
      a.t = __dadd_rn(a.t, o.t);
      for (int j = 0; j < NQ; ++j) a.q[j] = __dadd_rn(a.q[j], o.q[j]);
      for (int j = 0; j < NX; ++j) a.x[j] = __dadd_rn(a.x[j], o.x[j]);
      for (int j = 0; j < NY; ++j) a.y[j] = __dadd_rn(a.y[j], o.y[j]);
    }
    if (dead) a.fill(NAN);
    a.store(ld, i, t_bar, q_bar, x_bar, y_bar);
  }
}

template <class S, class P>
__device__ __forceinline__ void qp_rollout_tape(long long N, long long ld, int steps, double dt, const double* t0,
                                                int t_stride, double* q, double* x, const double* y, double vmax_q,
                                                double vmax_x, double* sol_last, int* n_failed, int max_iter,
                                                double* tape_q, double* tape_x, double* tape_sol, int* tape_status,
                                                unsigned* tape_active) {
  rollout_tape<S, QpRolloutState<S, P>>(N, ld, steps, dt, t0, t_stride, q, x, y, vmax_q, vmax_x, sol_last, n_failed,
                                        max_iter, tape_q, tape_x, tape_sol, tape_status, tape_active);
}

template <class S, class P>
__device__ __forceinline__ void nlp_rollout_tape(long long N, long long ld, int steps, double dt, const double* t0,
                                                 int t_stride, double* q, double* x, const double* y, double vmax_q,
                                                 double vmax_x, double* sol_last, int* n_failed, int max_iter,
                                                 double* tape_q, double* tape_x, double* tape_sol, int* tape_status,
                                                 unsigned* tape_active) {
  rollout_tape<S, NlpRolloutState<S, P>>(N, ld, steps, dt, t0, t_stride, q, x, y, vmax_q, vmax_x, sol_last, n_failed,
                                         max_iter, tape_q, tape_x, tape_sol, tape_status, tape_active);
}

template <class S>
__device__ __forceinline__ void qp_rollout_vjp(long long N, long long ld, int steps, double dt, const double* t0,
                                               int t_stride, const double* y, double vmax_q, double vmax_x,
                                               const double* tape_q, const double* tape_x, const double* tape_sol,
                                               const int* tape_status, const unsigned* tape_active,
                                               const double* q_bar_K, const double* x_bar_K, const double* sol_bar,
                                               double* t_bar, double* q_bar, double* x_bar, double* y_bar) {
  rollout_vjp<S, QpFace<S>>(N, ld, steps, dt, t0, t_stride, y, vmax_q, vmax_x, tape_q, tape_x, tape_sol, tape_status,
                            tape_active, q_bar_K, x_bar_K, sol_bar, t_bar, q_bar, x_bar, y_bar);
}

template <class S>
__device__ __forceinline__ void nlp_rollout_vjp(long long N, long long ld, int steps, double dt, const double* t0,
                                                int t_stride, const double* y, double vmax_q, double vmax_x,
                                                const double* tape_q, const double* tape_x, const double* tape_sol,
                                                const int* tape_status, const unsigned* tape_active,
                                                const double* q_bar_K, const double* x_bar_K, const double* sol_bar,
                                                double* t_bar, double* q_bar, double* x_bar, double* y_bar) {
  rollout_vjp<S, NlpAdjointFace<S>>(N, ld, steps, dt, t0, t_stride, y, vmax_q, vmax_x, tape_q, tape_x, tape_sol, tape_status,
                             tape_active, q_bar_K, x_bar_K, sol_bar, t_bar, q_bar, x_bar, y_bar);
}

}  // namespace clik
