/* clik.h — C ABI of the B200 batched CLIK controller-step engine (libclik_b200.so).
 *
 * The reference (mahaarbo/casclik) has no C ABI of its own: its controller step is Python calling
 * CasADi.  What it *effectively* binds per skill is CasADi's generated-code ABI — one JIT-compiled
 * function per mode, `cs.Function(..., {"jit": True})` at
 *     casclik/controllers/pseudo_inverse.py:476-483   (cntrl_var_<mode>)
 *     casclik/controllers/reactive_qp.py:283-294      (H_func / A_func / Blb_func / Bub_func)
 * plus the conic plugin call `cs.conic("solver", "qpoases", ...)` at reactive_qp.py:256-260 and
 * its invocation at :493 / :512-513.  Each entry point below names the reference call it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross this boundary;
 *   - batch arrays are structure-of-arrays: coordinate j of instance i is at  a[j*N + i];
 *   - `*_step` entry points take DEVICE pointers and are asynchronous on `stream` (a cudaStream_t
 *     passed as void*; NULL = legacy default stream); no hidden host synchronisation;
 *   - `*_step_host` entry points take HOST pointers, run H2D copy -> kernel -> D2H copy in a
 *     chunked two-stream pipeline and return when the outputs are in host memory;
 *   - errors are return codes (0 = CLIK_OK) + clik_last_error(); per-instance outcomes are
 *     status arrays (mode = -1, QP status), never exceptions;
 *   - a clik_skill is immutable after load and may be used from several host threads as long as
 *     each call uses its own stream and buffers.
 */
#ifndef CLIK_H_
#define CLIK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CLIK_ABI_VERSION 2

typedef enum {
  CLIK_OK = 0,
  CLIK_ERR_INVALID = 1,  /* bad argument (NULL where data is required, size mismatch) */
  CLIK_ERR_CUDA = 2,     /* CUDA runtime error, text in clik_last_error() */
  CLIK_ERR_IMAGE = 3,    /* cubin does not contain the kernels the descriptor promises */
  CLIK_ERR_NOGPU = 4     /* no CUDA device / driver */
} clik_status;

/* Per-instance QP outcome written to `status[i]` by clik_qp_step / clik_qp_dense.
 * The reference surfaces 1/2 as a RuntimeError out of `self.solver(...)` (reactive_qp.py:493). */
#define CLIK_QP_SOLVED 0
#define CLIK_QP_MAXITER 1
#define CLIK_QP_INFEASIBLE 2
#define CLIK_QP_INVALID 4 /* non-finite data or solution (NaN input, non-positive cost weight); 3 is internal */

/* Per-instance NLP outcome written to `status[i]` by clik_nlp_step*: CLIK_QP_SOLVED, CLIK_QP_MAXITER (SQP
 * iteration cap or the cap of a subproblem), CLIK_QP_INFEASIBLE, CLIK_QP_INVALID (also a non-finite cost,
 * gradient or Hessian at an iterate, or a Hessian no tried shift makes positive definite), or: */
#define CLIK_NLP_STALLED 5 /* the line search found no sufficient decrease of the cost */

/* Sizes of a compiled skill; must match the constants baked into the cubin (checked at load).
 * An image of the NLP controller (manifest flag 256) loads with has_pinv = has_qp = 0; qp_n / qp_m then
 * carry the NLP's decision variables and constraint rows. */
typedef struct {
  int32_t abi_version; /* CLIK_ABI_VERSION */
  int32_t device;      /* CUDA device ordinal the skill lives on */
  int32_t n_robot;     /* SkillSpecification.n_robot_var */
  int32_t n_virtual;   /* n_virtual_var (0 if the skill has none) */
  int32_t n_input;     /* n_input_var actually read by the kernels (0 if unused) */
  int32_t n_slack;     /* n_slack_var */
  int32_t n_modes;     /* 2^S for S SetConstraints; 1 if S = 0 */
  int32_t has_pinv;    /* cubin exports clik_pinv_kernel */
  int32_t has_qp;      /* cubin exports clik_qp_kernel */
  int32_t qp_n;        /* QP variables  nx = n_robot + n_virtual + n_slack */
  int32_t qp_m;        /* QP rows */
  int32_t block_threads; /* launch block size the kernels were tuned for (0 = default 128) */
} clik_skill_desc;

typedef struct clik_skill clik_skill;

/* Load the sm_100a cubin produced by the expression compiler for one skill.
 * Replaces the reference's per-mode JIT + dlopen (pseudo_inverse.py:474-483,
 * reactive_qp.py:283-298): one image holds every mode and both controllers' kernels. */
clik_status clik_skill_load(const void* cubin, size_t len, const clik_skill_desc* desc,
                            clik_skill** out);
void clik_skill_free(clik_skill* skill);

/* PseudoInverseController.solve (pseudo_inverse.py:512-556) for N instances.
 *   t      [N] (t_stride = 1) or [1] (t_stride = 0)          time_var
 *   q      [n_robot * N]                                      robot_var
 *   x      [n_virtual * N] or NULL when n_virtual = 0         virtual_var
 *   y      [n_input * N]   or NULL when n_input = 0           input_var
 *   qdot   [n_robot * N]   out                                cntrl_rob
 *   xdot   [n_virtual * N] out, or NULL when n_virtual = 0    cntrl_virt
 *   mode   [N] out, may be NULL                               current_mode (-1: none admissible, velocities 0)
 * Skills whose activation map has a run-time tail (more than 8 modes on dense sets) run, when `mode` is
 * given, as two launches: the statically compiled modes for every instance (one thread per instance),
 * then the rest of the map for the instances those rejected, CLIK_GROUP lanes per instance
 * (csrc/clik_pinv_group.cuh), handed over through mode[] with the transient value -2.  With mode == NULL
 * or CLIK_PINV_SPLIT=0: one launch.  CLIK_PINV_GROUP=1 runs whole batches in the sub-warp mapping. */
clik_status clik_pinv_step(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                           const double* q, const double* x, const double* y, double* qdot,
                           double* xdot, int32_t* mode, void* stream);

/* The same step for one SHARD of a larger batch, without repacking: N instances are processed, rows of
 * every array are `ld` elements apart (ld >= N), and every pointer (t when t_stride = 1, q, x, y, qdot,
 * xdot, mode) already points at the shard's first instance.  clik_pinv_step(..N..) == clik_pinv_step_ld(..N, N..).
 * This is how one batch is split over the GPUs of a box (BASELINE.json north_star: "sharded across the
 * 8 GPUs ... no NCCL on the hot path"): shard k of a mapped host batch runs on device k in place. */
clik_status clik_pinv_step_ld(const clik_skill* skill, int64_t N, int64_t ld, const double* t,
                              int32_t t_stride, const double* q, const double* x, const double* y,
                              double* qdot, double* xdot, int32_t* mode, void* stream);

/* The simulation loop CASCLIK users run around solve() (examples/notebooks/ur5_moe2016_example2.ipynb
 * cell 12, raw lines :535-549), `steps` controller steps per instance on the device:
 *     v = solve(t0 + k*dt, q, x, y);  v = clip(v, +-max_speed);  q += v_rob*dt;  x += v_virt*dt
 *   q, x            in/out: state at t0 on entry, state after `steps` steps on return
 *   max_robot_speed, max_virtual_speed   clip limits (pass INFINITY for none)
 *   qdot_last, xdot_last, mode_last      out, may be NULL: the last (clipped) command and its mode
 *   n_failed        out, may be NULL: number of steps in which no mode was admissible */
clik_status clik_pinv_rollout(const clik_skill* skill, int64_t N, int32_t steps, double dt,
                              const double* t0, int32_t t_stride, double* q, double* x,
                              const double* y, double max_robot_speed, double max_virtual_speed,
                              double* qdot_last, double* xdot_last, int32_t* mode_last,
                              int32_t* n_failed, void* stream);

/* ReactiveQPController.solve (reactive_qp.py:461-528) for N instances.
 *   x0     [qp_n * N] primal warm start or NULL (as the reference's x0=, :495-513): used to guess
 *          the working set (rows that sit on a bound at x0); never changes the answer
 *   active0 [2 * N] or NULL: explicit working-set guess in the format of `active` (e.g. the
 *          previous step's output; may alias `active`); takes precedence over x0
 *   sol    [qp_n * N] out: [robot vel; virtual vel; slack]
 *   status [N] out, may be NULL: CLIK_QP_*.  With a status array, skills built with the working-set
 *          prediction run as two launches (prediction for every instance, then the full solver on the
 *          instances it could not certify, handed over through status[] with the transient value 3);
 *          with status == NULL, or CLIK_QP_SPLIT=0 in the environment, as one launch.  Same results.
 *   active [2 * N] out, may be NULL: active[i] bit r = row r at its upper bound,
 *          active[N + i] bit r = row r at its lower bound (rows >= 32 are not reported)
 *   max_iter <= 0 selects the default cap 10 * (qp_n + qp_m). */
clik_status clik_qp_step(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                         const double* q, const double* x, const double* y, const double* x0,
                         const uint32_t* active0, double* sol, int32_t* status, uint32_t* active,
                         int32_t max_iter, void* stream);

/* Shard variant of clik_qp_step (see clik_pinv_step_ld): active[i] / active[ld + i]. */
clik_status clik_qp_step_ld(const clik_skill* skill, int64_t N, int64_t ld, const double* t,
                            int32_t t_stride, const double* q, const double* x, const double* y,
                            const double* x0, const uint32_t* active0, double* sol, int32_t* status,
                            uint32_t* active, int32_t max_iter, void* stream);

/* The same simulation loop with the QP controller (see clik_pinv_rollout).  A step whose QP is not
 * solved applies zero velocity and is counted in n_failed (the reference would raise there).
 *   sol_last [qp_n * N] out, may be NULL: solution of the last step (robot part clipped) */
clik_status clik_qp_rollout(const clik_skill* skill, int64_t N, int32_t steps, double dt,
                            const double* t0, int32_t t_stride, double* q, double* x, const double* y,
                            double max_robot_speed, double max_virtual_speed, double* sol_last,
                            int32_t* n_failed, int32_t max_iter, void* stream);

/* The conic call itself, `solver(h=H, a=A, lba=lb, uba=ub[, x0=])` (reactive_qp.py:493), for N
 * numeric problems of one shape: min 1/2 x' diag(h) x, lb <= A x <= ub.
 *   h [nx * N], A [(m * nx) * N] row-major per instance (entry (r, c) at A[(r*nx + c)*N + i]),
 *   lb, ub [m * N].  Limits: nx <= 32, m <= 64 (two capacity tiers: up to 16 x 32 and up to 32 x 64; the
 *   working set is reported for the first 32 rows).  +-inf bounds are allowed. */
clik_status clik_qp_dense(int32_t device, int64_t N, int32_t nx, int32_t m, const double* h,
                          const double* A, const double* lb, const double* ub, const double* x0,
                          double* sol, int32_t* status, uint32_t* active, int32_t max_iter,
                          void* stream);

/* ReactiveNLPController.solve (the reference's cs.nlpsol / IPOPT call, reactive_nlp.py:469-534) for N
 * instances of an NLP image: min F(x) s.t. lb <= A x <= ub with the QP's rows, by SQP with the exact Hessian,
 * one instance per thread.
 *   x0     [qp_n * N] start point of the iteration, or NULL (start at 0); the first subproblem restores
 *          feasibility from it
 *   sol    [qp_n * N] out: [robot vel; virtual vel; slack]
 *   status [N] out, may be NULL: CLIK_QP_* / CLIK_NLP_STALLED
 *   iters  [N] out, may be NULL: SQP iterations (subproblems solved)
 *   active [2 * N] out, may be NULL: working set of the last subproblem, format of clik_qp_step
 *   max_iter <= 0 selects the default SQP cap 50.
 * Solved (0) means |p|_inf * max(1, delta) <= tol * (1 + |x|_inf) for the last SQP step p (delta: the shift that
 * made the Hessian positive definite, tol compiled into the image, default 1e-10), or a step with
 * |p|_inf <= 100 * tol * (1 + |x|_inf) that left the cost unchanged within its rounding (1e-15 relative). */
clik_status clik_nlp_step(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                          const double* q, const double* x, const double* y, const double* x0, double* sol,
                          int32_t* status, int32_t* iters, uint32_t* active, int32_t max_iter, void* stream);

/* Shard variant of clik_nlp_step (see clik_pinv_step_ld): N instances in place, rows `ld` elements apart
 * (ld >= N), every pointer (t when t_stride = 1, q, x, y, x0, sol, status, iters, active) already at the shard's
 * first instance; active[i] / active[ld + i].  clik_nlp_step(..N..) == clik_nlp_step_ld(..N, N..). */
clik_status clik_nlp_step_ld(const clik_skill* skill, int64_t N, int64_t ld, const double* t,
                             int32_t t_stride, const double* q, const double* x, const double* y,
                             const double* x0, double* sol, int32_t* status, int32_t* iters,
                             uint32_t* active, int32_t max_iter, void* stream);

/* The same call on HOST pointers, synchronous (the chunked pipeline or, on page-locked buffers, the kernel
 * on the mapped memory, as clik_qp_step_host).  Bit-identical to clik_nlp_step. */
clik_status clik_nlp_step_host(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                               const double* q, const double* x, const double* y, const double* x0,
                               double* sol, int32_t* status, int32_t* iters, uint32_t* active,
                               int32_t max_iter);

/* One instance, HOST pointers (the reference's single solve() call), synchronous, as clik_qp_solve_one. */
clik_status clik_nlp_solve_one(const clik_skill* skill, double t, const double* q, const double* x,
                               const double* y, const double* x0, double* sol, int32_t* status,
                               int32_t* iters, uint32_t* active, int32_t max_iter);

/* The simulation loop with the NLP controller (see clik_qp_rollout): every step starts from the previous
 * step's solution; a step that is not solved applies zero velocity, is counted in n_failed, and the next
 * step starts from 0.
 *   sol_last [qp_n * N] out, may be NULL: solution of the last step (robot / virtual parts clipped) */
clik_status clik_nlp_rollout(const clik_skill* skill, int64_t N, int32_t steps, double dt,
                             const double* t0, int32_t t_stride, double* q, double* x, const double* y,
                             double max_robot_speed, double max_virtual_speed, double* sol_last,
                             int32_t* n_failed, int32_t max_iter, void* stream);

/* Host-buffer variants (same argument meaning, HOST pointers, synchronous).  Pageable memory goes
 * through a chunked H2D / kernel / D2H pipeline on internal streams; if every buffer is page-locked
 * (cudaHostAlloc / cudaHostRegister, torch pin_memory()) the kernel runs directly on the mapped
 * host memory instead (CLIK_ZERO_COPY=0 disables this): one kernel per call (no fast + tail hand-over
 * through host memory), launched as a grid-stride grid of 2 CTAs per SM so that the reads the host sees
 * stay nearly sequential (CLIK_ZC_CTAS_PER_SM overrides, 0 = one CTA per 128 instances).  Results are
 * bit-identical to the device-pointer entry points on every path. */
clik_status clik_pinv_step_host(const clik_skill* skill, int64_t N, const double* t,
                                int32_t t_stride, const double* q, const double* x,
                                const double* y, double* qdot, double* xdot, int32_t* mode);
clik_status clik_qp_step_host(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                              const double* q, const double* x, const double* y, const double* x0,
                              const uint32_t* active0, double* sol, int32_t* status, uint32_t* active,
                              int32_t max_iter);

/* One instance, HOST pointers to its vectors (t by value): the reference's solve() call itself
 * (pseudo_inverse.py:512-556, reactive_qp.py:461-528), synchronous.  The instance travels through a
 * page-locked device-mapped slot owned by the skill (no allocation, copy engine or pointer query per call):
 * launch + wait, ~10 us.   active[2] = {upper mask, lower mask}. */
clik_status clik_pinv_solve_one(const clik_skill* skill, double t, const double* q, const double* x,
                                const double* y, double* qdot, double* xdot, int32_t* mode);
clik_status clik_qp_solve_one(const clik_skill* skill, double t, const double* q, const double* x,
                              const double* y, const double* x0, double* sol, int32_t* status,
                              uint32_t* active, int32_t max_iter);

/* The same single-instance steps with the constraint multipliers of the result (see clik_qp_duals):
 * lam [qp_m] out, or NULL.  The step and the multiplier kernel are launched back to back on the skill's
 * stream with one wait.  clik_qp_solve_one / clik_nlp_solve_one are these calls with lam = NULL, with
 * bit-identical results.  A non-NULL lam on a skill with more than 32 rows fails with CLIK_ERR_INVALID. */
clik_status clik_qp_solve_one_lam(const clik_skill* skill, double t, const double* q, const double* x,
                                  const double* y, const double* x0, double* sol, int32_t* status,
                                  uint32_t* active, int32_t max_iter, double* lam);
clik_status clik_nlp_solve_one_lam(const clik_skill* skill, double t, const double* q, const double* x,
                                   const double* y, const double* x0, double* sol, int32_t* status,
                                   int32_t* iters, uint32_t* active, int32_t max_iter, double* lam);

/* Constraint multipliers of a step's output (the reference's lam_a of cs.conic, lam_g of cs.nlpsol), for N
 * instances: the inputs of the step (t, q, x, y as clik_qp_step / clik_nlp_step) and its outputs
 *   sol [qp_n * N], status [N], active [2 * N]   (all required)
 *   lam [qp_m * N] out: lam[r*N + i], CasADi's sign convention (> 0 at an upper bound, < 0 at a lower bound,
 *       any sign on an equality row), 0 on the rows outside the working set.
 * lam_W = argmin |D^1/2 (g + A_W' lam)| on the working set W of `active`, by modified Gram-Schmidt QR: for the QP
 * g = H x and D = H^-1 (exact stationarity of the face problem), for the NLP g = grad F(x) and D = I.  Every entry
 * of instance i is NaN when status[i] is not 0 (solved), or when the rows of W are linearly dependent (a QR pivot
 * below 1e-12 times the largest column norm).  One thread per instance.  The working-set masks describe rows
 * below 32 only: a skill with more than 32 rows has no multiplier kernel and the call fails with
 * CLIK_ERR_INVALID, "multipliers need at most 32 constraint rows".  clik_qp_duals takes QP images,
 * clik_nlp_duals NLP images.  Device pointers, asynchronous on `stream`; the _host forms take host arrays and
 * are synchronous (zero copy on page-locked buffers, else the chunked pipeline), with bit-identical results. */
clik_status clik_qp_duals(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                          const double* q, const double* x, const double* y, const double* sol,
                          const int32_t* status, const uint32_t* active, double* lam, void* stream);
clik_status clik_nlp_duals(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                           const double* q, const double* x, const double* y, const double* sol,
                           const int32_t* status, const uint32_t* active, double* lam, void* stream);
clik_status clik_qp_duals_host(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                               const double* q, const double* x, const double* y, const double* sol,
                               const int32_t* status, const uint32_t* active, double* lam);
clik_status clik_nlp_duals_host(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                                const double* q, const double* x, const double* y, const double* sol,
                                const int32_t* status, const uint32_t* active, double* lam);

/* Reverse-mode derivative (vector-Jacobian product) of a step's output, for N instances.  theta = (t, q, x, y) of
 * instance i; its step returned x* = sol and the working set W of `active`.  On W the step solves
 *   r1 = g(x, theta) + A_W(theta)' lam_W = 0   (QP: g = H(theta) x;  NLP: g = grad F(x, theta))
 *   r2 = A_W(theta) x - b_W(theta)       = 0   (b_r = ub_r for an upper bit, lb_r for a lower bit)
 * For the cotangent xb = sol_bar[:, i] the adjoint system [[M, A_W'], [A_W, 0]] [u; v] = [xb; 0] (M = H, or
 * grad^2 F(x*) for the NLP) gives theta_bar = -grad_theta (u'(g + A' lam) + v'(A_W x* - b_W)) with x*, lam, u, v
 * held fixed: (d(x*)/d(theta))' xb for the face problem of W.  It is the derivative of the step where strict
 * complementarity holds; where a row of W has lam = 0 it is the one-sided derivative that keeps W.  lam is
 * computed inside the kernel as clik_qp_duals / clik_nlp_duals compute it.  Adjoint solve: QP v = argmin
 * |D^1/2 (-xb + A_W' v)| with D = H^-1, u = D (xb - A_W' v); NLP grad^2 F(x*) = L L' (no shift), the same
 * least-squares solve on the columns L^-1 a_r, u = L^-T L^-1 (xb - A_W' v).
 *   inputs:  t, q, x, y as clik_qp_step / clik_nlp_step; sol [qp_n * N], status [N], active [2 * N] of the step;
 *            sol_bar [qp_n * N] the cotangent of sol (all required)
 *   outputs: t_bar [N] (per instance, also when t_stride = 0: the caller sums it for a shared t),
 *            q_bar [n_robot * N], x_bar [n_virtual * N], y_bar [n_input * N] (x_bar / y_bar may be NULL when the
 *            size is 0)
 * Rules: an instance whose cotangent column is all zeros gets exactly 0, whatever its status; otherwise every
 * output of the instance is NaN when status[i] is not 0, when A_W is rank-deficient (the tests of clik_qp_duals)
 * or, for the NLP, when a Cholesky pivot of grad^2 F(x*) is at or below 1e-12 max(1, max_j |H_jj|), the pivot threshold
 * of the step itself (a Hessian that is singular or indefinite to working precision).
 * The kernel is in images built with emit_skill(..., vjp=True) (manifest o[19]) only, and only for skills with
 * 1..32 constraint rows: other images, and a NULL skill, fail with CLIK_ERR_INVALID.  Device pointers only, row
 * stride N, asynchronous on `stream`; one thread per instance. */
clik_status clik_qp_vjp(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                        const double* q, const double* x, const double* y, const double* sol,
                        const int32_t* status, const uint32_t* active, const double* sol_bar, double* t_bar,
                        double* q_bar, double* x_bar, double* y_bar, void* stream);
clik_status clik_nlp_vjp(const clik_skill* skill, int64_t N, const double* t, int32_t t_stride,
                         const double* q, const double* x, const double* y, const double* sol,
                         const int32_t* status, const uint32_t* active, const double* sol_bar, double* t_bar,
                         double* q_bar, double* x_bar, double* y_bar, void* stream);

/* One host batch over several GPUs of the box: `skills[k]` is the same cubin loaded on device k
 * (clik_skill_load with desc.device = k); the batch is cut into n_skills contiguous shards (sizes differ
 * by at most one, shard k = [k*N/n .. )), each shard runs on its device from its own host thread (zero
 * copy on page-locked buffers — the SMs of device k read/write only shard k of the host arrays over that
 * device's PCIe link — or the chunked pipeline on pageable ones), and the call returns when every
 * result is in the caller's host arrays: the "final host gather" of the north star, with no collective
 * and no intermediate copy.  Results are bit-identical to the single-device call.  The handles stay owned by
 * the caller; several of them may live on one device (their shards then share it).  The NLP form takes the
 * arguments of clik_nlp_step_host; clik_*_step_host(skill, ...) is clik_*_step_host_multi(&skill, 1, ...), so a
 * NULL skill there fails with CLIK_ERR_INVALID, "no skill handles". */
clik_status clik_pinv_step_host_multi(const clik_skill* const* skills, int32_t n_skills, int64_t N,
                                      const double* t, int32_t t_stride, const double* q,
                                      const double* x, const double* y, double* qdot, double* xdot,
                                      int32_t* mode);
clik_status clik_qp_step_host_multi(const clik_skill* const* skills, int32_t n_skills, int64_t N,
                                    const double* t, int32_t t_stride, const double* q, const double* x,
                                    const double* y, const double* x0, const uint32_t* active0,
                                    double* sol, int32_t* status, uint32_t* active, int32_t max_iter);
clik_status clik_nlp_step_host_multi(const clik_skill* const* skills, int32_t n_skills, int64_t N,
                                     const double* t, int32_t t_stride, const double* q, const double* x,
                                     const double* y, const double* x0, double* sol, int32_t* status,
                                     int32_t* iters, uint32_t* active, int32_t max_iter);

/* Overlap of launches on one stream (programmatic dependent launch, sm_90+; replaces nothing in the
 * reference — its loop is sequential, casclik/controllers/pseudo_inverse.py:512-556 — it is the batched
 * counterpart of calling solve() back to back).
 *   0  plain stream order: a launch starts when everything before it on the stream has completed;
 *   1  (default) the second launch of a two-launch step (QP fast + tail pass, pinv fast + group pass) is
 *      scheduled while the first drains and waits on the device for it to complete before it reads —
 *      same results, same ordering towards everything else on the stream;
 *   2  additionally the FIRST launch of every clik_pinv_step* / clik_qp_step* call may begin while the
 *      previous kernel on the stream is still draining (its last CTAs running).  The caller thereby declares
 *      that the call does not read what the previous launch on the stream writes and does not write what it
 *      reads (a stream of independent batches).  Kernels still COMPLETE in stream order, so events,
 *      copies and any kernel launched without this level keep their usual meaning.  Never use it when step
 *      k+1 consumes step k's output through device memory (use the rollout entry points for closed loops).
 * CLIK_PDL=<level> in the environment sets the level at load time. */
clik_status clik_skill_set_overlap(clik_skill* skill, int32_t level);
int32_t clik_skill_get_overlap(const clik_skill* skill);

/* Input staging of clik_pinv_step* on device-resident batches: on = the TMA-staged persistent kernel
 * (one CTA per resident slot walks tiles of 128 instances; the input rows the skill reads are brought into
 * shared memory by bulk async copies that complete on an mbarrier, two tiles ahead of the arithmetic), off
 * (default) = one CTA per 128 instances loading its own inputs.  Same results to the bit.  Staging pays for
 * HBM-leaning skills when batches alternate over two streams (+3 % on the tracking skill) and costs 1-3 % when
 * launches run one after the other; it needs 16-byte aligned rows (even ld, aligned bases), otherwise the call
 * silently uses the plain kernel.  CLIK_ERR_INVALID if the image has no staged kernel (skills with a
 * two-launch step, more than 16 input rows or more than 8 task rows). */
clik_status clik_skill_set_staging(clik_skill* skill, int32_t on);
int32_t clik_skill_get_staging(const clik_skill* skill);

/* Launch geometry chosen at load time (for reporting). */
clik_status clik_skill_launch_info(const clik_skill* skill, int32_t which /*0 pinv, 1 qp, 2 pinv TMA-staged, 3 qp fast pass, 4 qp tail pass, 5 pinv fast pass, 6 pinv group pass, 7 qp tail pass capped to 4 CTAs/SM (large batches)*/,
                                   int32_t* grid, int32_t* block, int32_t* regs_per_thread,
                                   int32_t* local_bytes_per_thread);

/* Measurement helpers used by bench.py (not part of the controller path):
 * sustained fp64 FMA throughput of the device in TFLOP/s (FMA = 2 flops), measured with
 * CUDA events over `iters` dependent-chain FMAs per thread on a full grid; and an L2 flush
 * (writes a buffer larger than L2). */
clik_status clik_measure_fp64_peak(int32_t device, int32_t iters, double* tflops);
clik_status clik_flush_l2(int32_t device, void* stream);

int32_t clik_device_count(void);
int32_t clik_abi_version(void);
const char* clik_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* CLIK_H_ */
