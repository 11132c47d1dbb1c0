// clik_duals.cuh — constraint multipliers of the QP and NLP controller steps at their returned point, one
// instance per thread, fp64, sm_100a.
//
// Both controllers return the primal solution x and the working set W of rows held at a bound (the two
// 32-bit masks of `active`).  The multipliers on W are the least-squares solution of stationarity in the
// metric D (positive diagonal):
//
//     lam_W = argmin |D^1/2 (g + A_W' lam)|,     lam = 0 off W
//
//   QP  (clik_qp.cuh):  g = H x, D = H^-1: exact stationarity of the face problem (z = sqrt(H) x coordinates,
//                       the coordinates the QP core works in);
//   NLP (clik_nlp.cuh): g = grad F(x), D = I.
//
// Modified Gram-Schmidt QR of the columns D^1/2 a_r (two orthogonalisation passes, as the QP core
// refactors its working set), then R lam = -Q' D^1/2 g: the condition number of A_W enters once, not squared
// as in the normal equations.  Sign convention of CasADi's lam_a / lam_g: lam > 0 at an upper bound, < 0 at a
// lower bound, any sign on an equality row; the unsigned solve gives it directly.  A rank-deficient A_W (a
// pivot below 1e-12 max_r |D^1/2 a_r|, or more rows than variables) has no unique multipliers: every entry is
// NaN, as for an instance that is not solved.
//
// The generated skill provides (codegen/emit.py) S::eval_qp (QP images) or S::eval_nlp_pre / S::eval_nlp_fgH
// (NLP images) and the input read masks; the masks describe rows below 32 only, so skills with more rows
// have no multiplier kernel.
#pragma once
#include <cmath>

#include "clik_nlp.cuh"

namespace clik {

// Working set of the masks up / lo: rows W[0..k) in ascending order, lam[r] = 0 for every row; false when more
// rows are held than there are variables (dependent).
template <int N, int M>
__device__ __forceinline__ bool working_set_rows(unsigned up, unsigned lo, int (&W)[N], int& k, double* lam) {
  static_assert(M <= 32, "the working-set masks describe rows below 32 only");
  k = 0;
  for (int r = 0; r < M; ++r) {
    lam[r] = 0.0;
    if (((up | lo) >> r) & 1u) {
      if (k < N) W[k] = r;
      ++k;
    }
  }
  return k <= N;
}

// QR step: Q holds k pre-scaled columns D^1/2 a_r (N entries each) on entry and their orthonormal basis on
// return, R (N x N, upper) the factor.  Modified Gram-Schmidt, two orthogonalisation passes; false when a
// pivot falls below 1e-12 max_r |D^1/2 a_r| (rank-deficient).
template <int N>
__device__ __forceinline__ bool working_set_qr(int k, double* Q, double* R) {
  double cmax = 0.0;
  for (int a = 0; a < k; ++a) {
    const double* col = &Q[a * N];
    double nrm = 0.0;
    for (int j = 0; j < N; ++j) nrm = fma(col[j], col[j], nrm);
    cmax = fmax(cmax, sqrt(nrm));
  }
  for (int a = 0; a < k; ++a) {
    double* col = &Q[a * N];
    for (int pass = 0; pass < 2; ++pass) {
      for (int l = 0; l < a; ++l) {
        double dt = 0.0;
        for (int j = 0; j < N; ++j) dt = fma(Q[l * N + j], col[j], dt);
        for (int j = 0; j < N; ++j) col[j] = fma(-dt, Q[l * N + j], col[j]);
        R[l * N + a] = (pass == 0) ? dt : R[l * N + a] + dt;
      }
    }
    double nrm = 0.0;
    for (int j = 0; j < N; ++j) nrm = fma(col[j], col[j], nrm);
    nrm = sqrt(nrm);
    if (!(nrm > 1e-12 * cmax)) return false;
    R[a * N + a] = nrm;
    const double inv = 1.0 / nrm;
    for (int j = 0; j < N; ++j) col[j] *= inv;
  }
  return true;
}

// Solve step: c = argmin |sg + (Q R) c| for the pre-scaled gradient sg = D^1/2 g, i.e. R c = -Q' sg
// (c = Q' b with b = -sg projected out column by column, two passes, then back substitution).  Writes
// lam[W[a]] = c[a].
template <int N>
__device__ __forceinline__ void working_set_solve(int k, const int* W, const double* Q, const double* R,
                                                  const double* sg, double* lam) {
  double c[N], b[N];
  for (int j = 0; j < N; ++j) b[j] = -sg[j];
  for (int a = 0; a < k; ++a) c[a] = 0.0;
  for (int pass = 0; pass < 2; ++pass) {
    for (int a = 0; a < k; ++a) {
      double dt = 0.0;
      for (int j = 0; j < N; ++j) dt = fma(Q[a * N + j], b[j], dt);
      for (int j = 0; j < N; ++j) b[j] = fma(-dt, Q[a * N + j], b[j]);
      c[a] += dt;
    }
  }
  for (int a = k - 1; a >= 0; --a) {
    double acc = c[a];
    for (int l = a + 1; l < k; ++l) acc = fma(-R[a * N + l], c[l], acc);
    c[a] = acc / R[a * N + a];
    lam[W[a]] = c[a];
  }
}

// A: M x N row-major, s = D^1/2 (diagonal), g: gradient; up / lo: working-set masks.  Writes lam[0..M);
// false (lam all NaN) when A_W is rank-deficient.
template <int N, int M>
__device__ __forceinline__ bool working_set_multipliers(const double* A, const double* s, const double* g,
                                                        unsigned up, unsigned lo, double* lam) {
  int W[N];
  double Q[N * N], R[N * N], sg[N];
  int k;
  bool ok = working_set_rows<N, M>(up, lo, W, k, lam);
  if (ok) {
    for (int a = 0; a < k; ++a)
      for (int j = 0; j < N; ++j) Q[a * N + j] = s[j] * A[W[a] * N + j];
    ok = working_set_qr<N>(k, Q, R);
  }
  if (!ok) {
    for (int r = 0; r < M; ++r) lam[r] = NAN;
    return false;
  }
  for (int j = 0; j < N; ++j) sg[j] = s[j] * g[j];
  working_set_solve<N>(k, W, Q, R, sg, lam);
  return true;
}

// Instance i's inputs, only the rows the generated program reads (masks RT, RQ, RX, RY of the image).
template <class S, unsigned RT, unsigned RQ, unsigned RX, unsigned RY>
__device__ __forceinline__ void duals_load(long long ld, long long i, const double* __restrict__ t, int t_stride,
                                           const double* __restrict__ q, const double* __restrict__ x,
                                           const double* __restrict__ y, double& tv, double (&qv)[S::NQ > 0 ? S::NQ : 1],
                                           double (&xv)[S::NX > 0 ? S::NX : 1], double (&yv)[S::NY > 0 ? S::NY : 1]) {
  tv = RT ? t[(long long)t_stride * i] : 0.0;
  for (int j = 0; j < S::NQ; ++j) qv[j] = row_read(RQ, j) ? q[(long long)j * ld + i] : 0.0;
  for (int j = 0; j < S::NX; ++j) xv[j] = row_read(RX, j) ? x[(long long)j * ld + i] : 0.0;
  for (int j = 0; j < S::NY; ++j) yv[j] = row_read(RY, j) ? y[(long long)j * ld + i] : 0.0;
}

// Multipliers of clik_qp_step's output (SoA, rows ld apart): lam[r*ld + i]; NaN unless status[i] is QP_OK.
template <class S>
__device__ __forceinline__ void qp_duals(long long N, long long ld, const double* __restrict__ t, int t_stride,
                                         const double* __restrict__ q, const double* __restrict__ x,
                                         const double* __restrict__ y, const double* __restrict__ sol,
                                         const int* __restrict__ status, const unsigned* __restrict__ active,
                                         double* __restrict__ lam) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    double l[S::QM];
    if (status[i] == QP_OK) {
      double tv, qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
      duals_load<S, S::QP_READ_T, S::QP_READ_Q, S::QP_READ_X, S::QP_READ_Y>(ld, i, t, t_stride, q, x, y, tv, qv, xv, yv);
      QpData<S> d;
      S::eval_qp(tv, qv, xv, yv, d);
      double s[S::QN], g[S::QN];
      for (int j = 0; j < S::QN; ++j) {
        s[j] = 1.0 / sqrt(d.h[j]);
        g[j] = d.h[j] * sol[(long long)j * ld + i];
      }
      working_set_multipliers<S::QN, S::QM>(d.A, s, g, active[i], active[ld + i], l);
    } else {
      for (int r = 0; r < S::QM; ++r) l[r] = NAN;
    }
    for (int r = 0; r < S::QM; ++r) lam[(long long)r * ld + i] = l[r];
  }
}

// Multipliers of clik_nlp_step's output: lam[r*ld + i]; NaN unless status[i] is 0 (solved).
template <class S>
__device__ __forceinline__ void nlp_duals(long long N, long long ld, const double* __restrict__ t, int t_stride,
                                          const double* __restrict__ q, const double* __restrict__ x,
                                          const double* __restrict__ y, const double* __restrict__ sol,
                                          const int* __restrict__ status, const unsigned* __restrict__ active,
                                          double* __restrict__ lam) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    double l[S::NM];
    if (status[i] == 0) {
      double tv, qv[S::NQ > 0 ? S::NQ : 1], xv[S::NX > 0 ? S::NX : 1], yv[S::NY > 0 ? S::NY : 1];
      duals_load<S, S::NLP_READ_T, S::NLP_READ_Q, S::NLP_READ_X, S::NLP_READ_Y>(ld, i, t, t_stride, q, x, y, tv, qv, xv,
                                                                                yv);
      NlpData<S> d;
      S::eval_nlp_pre(tv, qv, xv, yv, d);
      double v[S::NN], g[S::NN], H[S::NN * (S::NN + 1) / 2], one[S::NN];
      for (int j = 0; j < S::NN; ++j) {
        v[j] = sol[(long long)j * ld + i];
        one[j] = 1.0;
      }
      S::eval_nlp_fgH(d.P, v, g, H);
      working_set_multipliers<S::NN, S::NM>(d.A, one, g, active[i], active[ld + i], l);
    } else {
      for (int r = 0; r < S::NM; ++r) l[r] = NAN;
    }
    for (int r = 0; r < S::NM; ++r) lam[(long long)r * ld + i] = l[r];
  }
}

}  // namespace clik
