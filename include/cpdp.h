/* cpdp.h — C ABI of the B200 CPDP gradient-iteration library (one shared object per model:
 * libcpdp_<model>.so, built from learning-from-sparse-demonstrations_b200/csrc/cpdp_lib.cu).
 *
 * The reference has no FFI: the path sits behind Python methods of COCSys.  Each entry point below replaces
 * the numerical body of one of them; the Python class lfsd_b200.CPDP.COCSys binds them with ctypes
 * (INTEGRATION.md shows the stub a reference maintainer would add).
 *
 * Conventions: all arrays are row-major IEEE fp64 DEVICE pointers owned by the caller unless marked (host);
 * n = states, m = controls, r = learnable parameters (cpdp_model_dims), B problems, N grid intervals,
 * S RK4 sub-steps per interval.  Calls are stream-ordered on `stream` (a cudaStream_t passed as void*) and return 0, a
 * negative argument-error code or a positive cudaError_t (cpdp_error_string).  The library keeps no device state between
 * calls (everything lives in caller-owned buffers) and no host state shared between threads: the only host variables are
 * thread-local (the launch error of the call in progress, and the round count behind cpdp_last_rounds), so host threads
 * driving different streams or devices do not interfere.  Numerical outcomes are reported per problem in status arrays,
 * never as return codes.
 */
#ifndef CPDP_H
#define CPDP_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

/* per-problem solver status written by cpdp_solve; CPDP_INFEASIBLE: x0 is not strictly inside a finite state bound of its problem,
 * or (bounds that depend on pdata) some component of the problem has lb(pdata) >= ub(pdata).  Set at the start, cold or warm;
 * every auxiliary mode skips such a problem and cpdp_pack_rows counts it as failed. */
enum { CPDP_RUNNING = 0, CPDP_CONVERGED = 1, CPDP_MAXITER = 2, CPDP_LINESEARCH = 3, CPDP_NUMERIC = 4, CPDP_INFEASIBLE = 5 };

/* Model dimensions compiled into this library (COCSys.n_state / n_control / n_auxvar, CPDP.py:17,22,36);
 * q = number of per-problem constants (pdata, e.g. a goal position), 0 for most models. */
int cpdp_model_dims(int* n, int* m, int* r, int* q);

/* Length of one packed Riccati node [upper-tri(P) | W] = n(n+1)/2 + n*r (internal table of auxSysSolver). */
int cpdp_riccati_state_dim(void);

/* Box bounds compiled into this library (COCSys.setStateVariable / setControlVariable bounds): lb[n+m], ub[n+m] host arrays,
 * states then controls, -1e20 / +1e20 where there is none.  Returns 1 when some bound is finite, 0 otherwise, and 2 when some
 * bound is an expression of the per-problem constants pdata (those entries read NaN; cpdp_eval_bounds gives their values).  A
 * bounded library's cpdp_solve runs a primal-dual interior-point (barrier) method and keeps the bound multipliers in the
 * workspace; with pdata bounds each problem uses its own, and a bound evaluating to +-1e20 or beyond is no bound for that problem. */
int cpdp_bounds(double* lb, double* ub);

/* Bounds of B problems: device arrays lb[B][n+m], ub[B][n+m] evaluated at pdata[B][q] (device; may be null when no bound depends
 * on it).  Any library: constant bounds are broadcast, unbounded components read -1e20 / +1e20.  -1: lb or ub null or B <= 0;
 * -8: pdata null although some bound depends on it. */
int cpdp_eval_bounds(const double* pdata, int B, double* lb, double* ub, void* stream);

/* Copy the bound multipliers z_L, z_U [B][N+1][n+m] (row N: the final state's entries; 0 where there is no bound) and the barrier
 * parameter mu[B] out of the workspace a bounded cpdp_solve left them in (get), or into it (set).  cpdp_aux mode 2 reads them
 * there, so a solution passed in from elsewhere is differentiated after a set.  Device arrays; -11 for an unbounded library. */
int cpdp_get_bound_multipliers(void* ws, size_t ws_bytes, int B, int N, int S, double* Zl, double* Zu, double* mu, void* stream);
int cpdp_set_bound_multipliers(void* ws, size_t ws_bytes, int B, int N, int S, const double* Zl, const double* Zu,
                               const double* mu, void* stream);

/* 1 if mode 1 (as-shipped BDF backward sweep) of cpdp_aux is compiled in; ints per row of `counters`. */
int cpdp_has_bdf(void);
int cpdp_num_counters(void);

/* Bytes of scratch the caller must provide to cpdp_solve / cpdp_aux for (B, N, S). */
size_t cpdp_workspace_bytes(int B, int N, int S);

/* Replaces COCSys.cocSolver (CPDP.py:92-198) for B problems: RK4 multiple-shooting NLP, all-zeros seed,
 * Newton-KKT with IPOPT's inertia correction and filter line search; with box bounds (cpdp_bounds) IPOPT's primal-dual
 * barrier method on the same recursion (z_L, z_U, mu: cpdp_get_bound_multipliers).
 *   x0[B][n]; theta[B][r] (theta_stride = r) or shared theta[r] (theta_stride = 0); T horizon;
 *   tol: KKT tolerance; max_iter: Newton iteration cap, 0..255 (the per-problem filter holds 256 corners; -10 otherwise);
 *   rounds > 0: launch exactly that many Newton rounds with no host synchronisation (CUDA-graph capturable);
 *   rounds = 0: poll the number of unconverged problems (one stream sync per round) and stop early.
 * Outputs X[B][N+1][n], U[B][N+1][m] (row N copies row N-1, CPDP.py:191), Lam[B][N+1][n] (= lam_g, CPDP.py:193),
 * status[B], iters[B]; optional kkt_out[B], cost_out[B]. */
int cpdp_solve(void* ws, size_t ws_bytes, int B, int N, int S, double T,
               const double* x0, const double* theta, int theta_stride, const double* pdata /* [B][q] or NULL */,
               double tol, int max_iter, int rounds,
               double* X, double* U, double* Lam, int* status, int* iters,
               double* kkt_out, double* cost_out, void* stream);

/* cpdp_solve started from a given trajectory instead of the all-zeros seed (warm start; the Newton iteration itself is the same).
 *   Xg[B][N+1][n], Ug[B][N+1][m], Lg[B][N+1][n]: the guess, e.g. the outputs of a previous call; they may alias X, U, Lam.
 *   Zlg, Zug[B][N+1][n+m]: bound multipliers of the guess (bounded models; both or NULL, meaning z = mu_init / slack).
 *   init_status[B] (may be NULL; may alias status): a problem whose entry is not CPDP_CONVERGED gets cpdp_solve's cold seed.
 *   shift 0: row k starts from guess row k; shift 1 (receding horizon): from guess row min(k+1, last row), i.e. X, Lam and the
 *   states' z repeat row N, U and the controls' z row N-1.  Either way X_0 = x0 and U_N = U_{N-1}.
 *   mu_init > 0: barrier parameter of a warm-started problem (bounded models; ignored otherwise).  A bounded model follows IPOPT's
 *   warm_start_init_point: the guess is pushed into the interior by 1e-3 (warm_start_bound_push / _frac), z = max(z, 1e-3).
 * Outputs and per-problem status as cpdp_solve; a converged guess of the same problem ends with iters = 0.  -12: shift not 0 or 1;
 * -13: mu_init <= 0 on a bounded library. */
int cpdp_solve_warm(void* ws, size_t ws_bytes, int B, int N, int S, double T,
                    const double* x0, const double* theta, int theta_stride, const double* pdata,
                    double tol, int max_iter, int rounds,
                    double* X, double* U, double* Lam, int* status, int* iters,
                    double* kkt_out, double* cost_out, void* stream,
                    const double* Xg, const double* Ug, const double* Lg, const double* Zlg, const double* Zug,
                    const int* init_status, int shift, double mu_init);

/* Newton rounds launched by the most recent cpdp_solve or cpdp_solve_warm of the calling thread (4 kernel launches per round + 2). */
int cpdp_last_rounds(void);

/* Replaces COCSys.auxSysSolver (CPDP.py:301-381) and the getloss_*corrections closures
 * (lib/QuadAlgorithm.py:616-639, Examples/rocket_groundtruth.py:45-70) for B problems.
 *   mode 0: backward Riccati sweep by RK45 with (rtol_b, atol_b)   [what COCSys_TimeVarying does, CPDP.py:740]
 *   mode 1: backward sweep by the BDF scheme of the as-shipped COCSys (CPDP.py:335), scipy defaults in rtol_b/atol_b
 *   forward sweep: RK45 with (rtol_f, atol_f) (CPDP.py:368; scipy defaults 1e-3 / 1e-6).
 *   mode 2 ("discrete"): no integrator -- Xa, Ua, loss and dtheta are the exact derivative of the discretised problem cpdp_solve
 *   solves, from the KKT system of the RK4 multiple-shooting NLP differentiated at (X, U, Lam) (a Riccati recursion over the
 *   stage derivatives; the tolerances are ignored, S must be > 0, counters stay 0).  aux_status 4 here: some Quu block of the
 *   recursion is not positive definite (the reduced Hessian at the point is not positive definite).
 *   Loss: W waypoints of D observed state components sel[D] (host ints); taus[B][W] (taus_stride = W) or shared
 *   taus[W] (stride 0); wp[B][W][D].  W = 0 skips the loss.
 * Outputs Xa[B][N+1][n*r] (dx/dtheta nodes), Ua[B][N+1][m*r], loss[B], dtheta[B][r] (reference convention:
 * dl_dy = y - wp, i.e. half the true gradient), aux_status[B] (0 ok, 1 step too small, 2 non-finite, 3 skipped
 * because the forward solve produced no trajectory, 4 singular Newton matrix, 5 a waypoint time outside [0, T] -- scipy's
 * interp1d raises there in the reference), counters[B][cpdp_num_counters()=6]
 * (backward rhs evals, backward steps, forward rhs evals, forward steps, backward LU factorisations, backward
 * Jacobian evaluations). */
int cpdp_aux(void* ws, size_t ws_bytes, int B, int N, int S, double T,
             const double* theta, int theta_stride, const double* pdata,
             const double* X, const double* U, const double* Lam, const int* solve_status,
             int mode, double rtol_b, double atol_b, double rtol_f, double atol_f,
             int W, int D, const int* sel /* host */, const double* taus, int taus_stride, const double* wp,
             double* Xa, double* Ua, double* loss, double* dtheta, int* aux_status, int* counters, void* stream);

/* cpdp_aux with the two sweeps selectable: phases 1 = backward Riccati sweep only (node table left in ws),
 * 2 = forward sweep + loss only (needs the table of a previous phase-1 call on the same ws), 3 = both.
 * Mode 2: phase 1 = stage derivatives + backward recursion (gains left in ws), phase 2 = rollout + loss. */
int cpdp_aux_phases(void* ws, size_t ws_bytes, int B, int N, int S, double T,
             const double* theta, int theta_stride, const double* pdata,
             const double* X, const double* U, const double* Lam, const int* solve_status,
             int mode, double rtol_b, double atol_b, double rtol_f, double atol_f,
             int W, int D, const int* sel /* host */, const double* taus, int taus_stride, const double* wp,
             double* Xa, double* Ua, double* loss, double* dtheta, int* aux_status, int* counters, void* stream, int phases);

/* Adjoint of mode 2: for cotangents Xbar[B][N+1][n] and Ubar[B][N+1][m] of the trajectory (either may be NULL, meaning zero; not
 * both), theta_bar[B][r] = sum_k (dX_k/dtheta)' Xbar_k + (dU_k/dtheta)' Ubar_k and x0_bar[B][n] (may be NULL) the same with
 * respect to x0, the exact derivatives of the discretised problem cpdp_solve solves (mode 2's), by one reverse sweep per problem
 * instead of r forward columns.  U_N = U_{N-1} (CPDP.py:191), so a cotangent on U_N acts on U_{N-1}.  Self-contained: it runs
 * mode 2's stage derivatives and backward recursion first (S > 0; bounded models read z_L, z_U, mu from the workspace as mode 2
 * does: cpdp_set_bound_multipliers).  aux_status[B] as in mode 2 (0 ok, 3 no usable trajectory, 4 Quu not positive definite).
 * Rows are zero where aux_status != 0 or solve_status (may be NULL) is not CPDP_CONVERGED.  Bit-identical per problem for any
 * batching.  Same workspace and argument-error codes as cpdp_aux. */
int cpdp_aux_adjoint(void* ws, size_t ws_bytes, int B, int N, int S, double T,
                     const double* theta, int theta_stride, const double* pdata,
                     const double* X, const double* U, const double* Lam, const int* solve_status,
                     const double* Xbar, const double* Ubar, double* theta_bar, double* x0_bar, int* aux_status, void* stream);

/* Bytes of the pdata workspace of cpdp_aux_adjoint_pd for B problems of N intervals (0 when the model has no per-problem
 * constants).  Separate from cpdp_workspace_bytes, which does not change. */
size_t cpdp_pdata_workspace_bytes(int B, int N);

/* cpdp_aux_adjoint plus pdata_bar[B][q] = sum_k (dX_k/dpdata)' Xbar_k + (dU_k/dpdata)' Ubar_k, the gradient with respect to the
 * per-problem constants (DESIGN.md §3.11).  The q constants ride along as q extra parameter columns of the same sweep; pd_ws
 * (cpdp_pdata_workspace_bytes(B, N) bytes, -3 if smaller) holds their stage derivatives and gains.  theta_bar and x0_bar are those
 * of cpdp_aux_adjoint; same zero-row rule and argument-error codes, plus -14 (the model has no per-problem constants) and -15 (the
 * library was built without the pdata derivatives, or n + m + r + q > 32).  When bounds depend on pdata, pdata_bar includes the
 * bounds' part, -(Sigma_L dlb/dpdata + Sigma_U dub/dpdata) in the differentiated barrier KKT system (DESIGN.md §3.12). */
int cpdp_aux_adjoint_pd(void* ws, size_t ws_bytes, void* pd_ws, size_t pd_ws_bytes, int B, int N, int S, double T,
                        const double* theta, int theta_stride, const double* pdata,
                        const double* X, const double* U, const double* Lam, const int* solve_status,
                        const double* Xbar, const double* Ubar, double* theta_bar, double* x0_bar, double* pdata_bar,
                        int* aux_status, void* stream);

/* FP64 FMA throughput probe used by bench.py for the roofline denominator: one kernel of `blocks` x 256 threads,
 * 8 independent chains of `iters` DFMAs per thread (flops = blocks*256*8*iters*2).  sink: >= 1 device double. */
int cpdp_dfma_probe(double* sink, int blocks, int iters, void* stream);

/* Cross-problem sum of [loss | dL/dtheta] rows in a fixed binary tree over the row index (bit-identical for any
 * sharding of the rows over GPUs once they are all-gathered).  scratch: nextpow2(B)*(1+r) doubles; out[1+r]. */
int cpdp_reduce(const double* loss, const double* dtheta, int B, double* scratch, double* out, void* stream);

/* Rows [loss | dL/dtheta | bad] (r + 2 doubles per problem): the unit of the one cross-GPU exchange of an iteration
 * (all-gather) -- bad = 1 when the problem's forward solve did not end CPDP_CONVERGED (solve_status may be NULL) or its
 * aux_status != 0, so that failures travel with the sum instead of disappearing into it (the reference never looks at
 * IPOPT's status, CPDP.py:183).  rows[B][r+2]. */
int cpdp_pack_rows(const double* loss, const double* dtheta, const int* solve_status, const int* aux_status, int B,
                   double* rows, void* stream);

/* Fixed binary-tree sum over the row index of B rows of C doubles (same tree as cpdp_reduce; bit-identical for any
 * sharding of the rows).  With cpdp_pack_rows rows: out = [sum loss | sum dL/dtheta | number of failed problems].
 * scratch: nextpow2(B)*C doubles; out[C]. */
int cpdp_reduce_rows(const double* rows, int B, int C, double* scratch, double* out, void* stream);

/* Learner step on the device: replaces the update rules, projection and stop rule of lib/QuadAlgorithm.py:239-257,
 * 454-578 so that a learning run is a stream of launches (CUDA-graph capturable).
 *   phase 0: theta_eval[r] <- evaluation point of the next gradient iteration (theta + mu*velocity for Nesterov,
 *            QuadAlgorithm.py:480; theta otherwise; theta when defer_close = 1, the second evaluation of
 *            true_loss_print_flag).
 *   phase 1: update theta from red = [loss | dL/dtheta | ...] in the reference's numpy association, theta[0] =
 *            max(theta[0], 1e-8), param_trace[it+1] = theta, loss_trace[it] = loss, it[0] += 1, it[1] = 1 (stop) unless
 *            loss > loss_stop and |dL| > grad_stop.  defer_close = 1 leaves the iteration open for a phase-2 call.
 *   phase 2: record loss / apply the stop rule with a second evaluation at the updated theta (QuadAlgorithm.py:490-492).
 *   method: 0 Vanilla, 1 Nesterov, 2 Adam, 3 Nadam, 4 AMSGrad.  Once it[1] != 0 (or it[0] == cap) phases 1/2 do nothing.
 *   theta[r], theta_eval[r], state[3][r] (zeroed by the caller), it[2] (zeroed), loss_trace[cap],
 *   param_trace[cap+1][r] (row 0 = initial theta, written by the caller): all device memory. */
int cpdp_optim_step(int phase, int method, double lr, double mu, double beta1, double beta2, double eps,
                    double loss_stop, double grad_stop, double* theta, double* theta_eval, double* state,
                    const double* red, int* it, double* loss_trace, double* param_trace, int cap, int defer_close,
                    void* stream);

const char* cpdp_error_string(int code);

/* "CPDP_BUILD_DIGEST=<sha1>" of the generated model header, kernel sources and compiler flags this library was built
 * from (the host package uses it to recognise an up-to-date prebuilt library). */
const char* cpdp_build_digest(void);

#ifdef __cplusplus
}
#endif
#endif
