/* tmpc.h -- C ABI of the B200-native batched tuned-MPC feedback solver.
 *
 * One shared library per compiled model (libtmpc_<model>.so), every library exporting exactly these symbols --
 * the same arrangement as the reference's only native solver path, where `Pmpc.generate` emits one shared
 * library per model and binds it with ctypes through an opaque capsule
 * (reference: external/acados/interfaces/acados_template/acados_template/acados_ocp_solver.py:752-801,
 *  `*_acados_create_capsule / *_acados_create / *_acados_solve / *_acados_free`; used from tunempc/pmpc.py:425-472).
 *
 * What each entry point replaces in the reference's Python hot path:
 *   tmpc_create / tmpc_set_tables   Pmpc.__init__ -> __construct_solver + __create_reference  (tunempc/pmpc.py:39-147, 162-369, 676-783)
 *   tmpc_reset                      Pmpc.reset / __set_initial_guess                          (tunempc/pmpc.py:858-865, 930-948)
 *   tmpc_step / tmpc_step_host      Pmpc.step -> Sqp.solve for B initial states at once       (tunempc/pmpc.py:371-423, tunempc/sqp_method.py:136-183)
 *   tmpc_plant_step                 F(x0=x, p=u)['xf'] in closed_loop_sim                     (tunempc/closed_loop_tools.py:102)
 *   tmpc_plant_jacobian             the first-order sensitivities of that integrator, for backpropagation through a closed loop
 *   tmpc_stage_log                  cost(x,u), h(x,u) logged per closed-loop sample            (tunempc/closed_loop_tools.py:64-65, 98-99)
 *   tmpc_get_*                      Pmpc.w_sol / g_sol / log / index properties               (tunempc/pmpc.py:1120-1142, 785-831)
 *
 * Conventions: return 0 = success, non-zero = API error (message via tmpc_last_error); numerical failures never
 * abort the batch, they are reported per instance in `status`.  All matrices row-major unless stated.  Pointers
 * named *_dev are device pointers on the handle's device, *_host are host pointers.  The caller owns every buffer
 * it passes; the library owns its workspace.  Calls on one handle are not re-entrant.  fp64 throughout.
 */
#ifndef TMPC_H
#define TMPC_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct tmpc_handle tmpc_handle;

/* per-instance status (SURVEY.md section 5 "failure detection") */
#define TMPC_OK 0              /* converged: infeasibility < tol and |grad L|_inf < tol (sqp_method.py:276-277)   */
#define TMPC_MAX_ITER 1        /* stopped at k == max_iter (sqp_method.py:281)                                     */
#define TMPC_QP_INFEASIBLE 2   /* QP infeasible / working set overflow (reference: CasADi conic raises)            */
#define TMPC_NOT_PD 3          /* reduced Hessian not positive definite (reference: AssertionError sqp_method.py:201) */
#define TMPC_NAN 4             /* non-finite iterate                                                                */
#define TMPC_WS_OVERFLOW 5     /* dual active set needed more than opts.max_working_set rows                        */
/* flag bits OR-ed into `flags` output */
#define TMPC_FLAG_GN_FALLBACK 1  /* >=1 iteration used the Gauss-Newton Hessian because the exact one was not PD on the null
                                    space of [equalities; rows active in the multipliers] -- exactly where the reference
                                    eigen-clips its reduced Hessian (sqp_method.py:345-376)                         */
#define TMPC_FLAG_GN_RESOLVE 4   /* >=1 QP fell back to the Gauss-Newton Hessian after releasing wrong-signed base rows
                                    (the reference's QP is non-convex there)                                        */
#define TMPC_FLAG_NONCONVEX_STEP 8 /* >=1 QP was non-convex once wrong-signed rows were released and was continued by an
                                    inertia-controlling primal active-set step (the reference's qpOASES: flipping bounds)   */
#define TMPC_FLAG_DAMPED 2       /* >=1 line-search backtrack (alpha < 1)                                           */

typedef struct {
  int32_t nx, nu;        /* must equal the compiled model's (checked) */
  int32_t nh;            /* rows of h(x,u) = C z + c >= 0 */
  int32_t nx_term;       /* rows of the terminal operator (selection of states) */
  int32_t N;             /* horizon */
  int32_t p;             /* period of the reference tables */
  int32_t ns;            /* slacks us of the nonlinear path constraints: rows g_k = h_nl(x,u) - us = 0 (tunempc/preprocessing.py:78-118,
                            pmpc.py:50-55,222-228,270-271); must equal the compiled model's (checked) */
  int32_t nsc;           /* soft-constraint slacks usc with the linear cost scost'usc (tunempc/preprocessing.py:120-155,
                            pmpc.py:57-62,230-233,338-339); must equal the compiled model's (checked) */
} tmpc_dims;
/* Stage variables z_k = (x, u, us, usc), nz = nx + nu + ns + nsc (pmpc.py:217-235); n_w = N*nz + nx.
 * g = [init(nx) | k < N: dyn_k(nx), g_k(ns), h_k(nh) | term(nx_term)], n_g = nx + N*(nx+ns+nh) + nx_term (pmpc.py:242-256).
 * h rows are linear in z: [h_lin(x,u) (+ usc on slacked rows); us; usc] >= 0 (preprocessing.py:110-112,150). */

typedef struct {
  int32_t hessian_exact;   /* 1: exact Lagrangian Hessian (pmpc.py:153 default), 0: gauss_newton (pmpc.py:327-333) */
  int32_t max_iter;        /* pmpc.py:155 (2000) */
  int32_t max_ls_iter;     /* sqp_method.py:57 (300) */
  double tol;              /* sqp_method.py:55 (1e-6) */
  double lam_tresh;        /* sqp_method.py:56 (1e-8) */
  double ls_step_factor;   /* sqp_method.py:58 (0.8) */
  double reg_tol;          /* sqp_method.py:54 (1e-8): pivot threshold of the reduced-Hessian PD test */
  double term_weight;      /* weight (relative to the largest Hessian diagonal entry) of the augmented-Lagrangian term the base
                              factorisation carries for the terminal rows; the rows themselves are enforced exactly through their
                              multipliers in the Schur complement, so the QP solution does not depend on it */
  int32_t max_working_set; /* rows the dual active set may ADD to the base rows of one QP (default 32, clipped to N*nh); the base rows
                              (terminal rows + rows active in the multipliers) live in the factorisation and do not count.
                              Overflow is reported per instance as status TMPC_WS_OVERFLOW, never as "infeasible" */
  int32_t economic;        /* 1: economic MPC -- stage cost = the compiled model's l(x,u) + scost'usc, exact Hessian forced
                              (pmpc.py:97-107, 173-183, 299-301, 338-339): H and the (x,u,us) entries of q are ignored (pass
                              zeros), the usc entries of q still carry scost; 0: tuned / tracking cost from the H, q tables
                              (mtools.py:43-57) */
} tmpc_opts;

void tmpc_default_opts(tmpc_opts* o);
/* compiled model: name, nx, nu, RK4 steps (0 for a discrete map), step length */
const char* tmpc_model_info(int32_t* nx, int32_t* nu, int32_t* rk_steps, double* dt);
/* slack dimensions the model library was compiled for (0, 0 for a model without nonlinear / soft constraints) */
void tmpc_model_slacks(int32_t* ns, int32_t* nsc);

int tmpc_create(tmpc_handle** h, const tmpc_dims* dims, const tmpc_opts* opts, int device);
void tmpc_destroy(tmpc_handle* h);
const char* tmpc_last_error(const tmpc_handle* h);

/* host pointers, copied.  wref (p*nz) | H (p*nz*nz) | q (p*nz) per phase; ref_du (p*n_g) dual reference window per
 * phase in g-order; C (nh*nz), c (nh); term_idx (nx_term); relax0 (nh) 1 = row dropped at stage 0 (pmpc.py:293-294:
 * h_x_idx + h_us_idx, the caller computes the lists with the reference's formulas).  With slacks the tables are nz wide:
 * the usc entries of wref and the usc rows / columns of H are zero (the reference's wref and H have none, pmpc.py:186-208)
 * and the usc entries of q carry scost (pmpc.py:338-339: J += scost'usc). */
int tmpc_set_tables(tmpc_handle* h, const double* wref, const double* H, const double* q, const double* ref_du,
                    const double* C, const double* c, const int32_t* term_idx, const int32_t* relax0);

/* size the workspace for B instances, phase index <- 0, warm start <- reference (pmpc.py:858-865, 930-942) */
int tmpc_reset(tmpc_handle* h, int64_t B);
int tmpc_get_index(const tmpc_handle* h, int64_t* index);

/* One batched Pmpc.step: X0_dev (B*nx) -> U0_dev (B*nu).  Optional outputs (may be NULL): W_dev (B*n_w) primal
 * solution, LAM_dev (B*n_g) multipliers, G_dev (B*n_g) constraint values at the solution, status/iter/flags (B).
 * Side effects as in the reference: index += 1, warm start <- shifted solution (pmpc.py:415-421, 867-906).
 * Runs on `cuda_stream` (cudaStream_t, NULL = default) and returns after the SQP loop has finished (the host reads two device
 * counters per SQP iteration); tmpc_step_async below is the stream-ordered, non-blocking form. */
int tmpc_step(tmpc_handle* h, const double* X0_dev, int64_t B, double* U0_dev, double* W_dev, double* LAM_dev,
              double* G_dev, int32_t* status_dev, int32_t* iter_dev, int32_t* flags_dev, void* cuda_stream);
/* The same step as a NON-BLOCKING call: returns at once, the SQP loop is driven by a host worker thread of the handle on an
 * internal stream.  Work the caller enqueued on `cuda_stream` BEFORE the call (the producer of X0_dev) is waited for on the
 * device; the outputs are complete -- visible to every stream -- once tmpc_wait has returned (it blocks the host and returns the
 * step's code, 0 = ok, message via tmpc_last_error).  Until then no other call on the handle except tmpc_busy; one step in
 * flight per handle.  Use: overlap host work or other handles (tuned and economic controller, several devices) with the solve.
 * A device-side hold of the caller's stream (cuStreamWaitValue32 on a ticket the worker releases) was tried and deadlocked on the
 * test box, see DESIGN.md section 1. */
int tmpc_step_async(tmpc_handle* h, const double* X0_dev, int64_t B, double* U0_dev, double* W_dev, double* LAM_dev,
                    double* G_dev, int32_t* status_dev, int32_t* iter_dev, int32_t* flags_dev, void* cuda_stream);
int tmpc_wait(tmpc_handle* h);
int tmpc_busy(tmpc_handle* h, int32_t* busy);
/* same call with HOST buffers (pinned or pageable): H2D of X0, solve, D2H of the requested outputs */
int tmpc_step_host(tmpc_handle* h, const double* X0_host, int64_t B, double* U0_host, double* W_host,
                   double* LAM_host, double* G_host, int32_t* status_host, int32_t* iter_host, int32_t* flags_host);

/* Feedback Jacobian J_b = du0*_b / dx0_b of the solutions of the last tmpc_step / tmpc_step_host / (tmpc_step_async + tmpc_wait),
 * the quantity the tuned controller is built to match (first-order equivalence with the economic controller).
 * Definition: at instance b's solution (w*, lam*) the held set A is every equality row (init, dynamics, nonlinear rows g, terminal
 * rows) plus every inequality row with lam* != 0, except the rows relax0 drops at stage 0.  J_b is the u_0 block of dw in
 *     [H  J_A'; J_A  0] [dw; dlam] = [0; e_j on the init rows],   j = 0 .. nx-1,
 * with H the exact Hessian of the Lagrangian and J_A the Jacobian of the held rows: the derivative of the solution map (implicit
 * function theorem) under strict complementarity, the active set held.
 * Layout: J[b*nu*nx + i*nx + j] = d u0_i / d x0_j (B x nu x nx, row-major); jstatus (B) per instance, values below.
 * Buffers: host memory if dst_is_host != 0, else device memory on the handle's device (runs on `cuda_stream`).  Returns after
 * its kernels have finished.  Leaves the warm start, the phase index, the log, counters and timing unchanged.
 * API errors: no step has finished since tmpc_create / tmpc_reset; a step is in flight; the handle uses the Gauss-Newton
 * Hessian (hessian_exact = 0 and not economic).  After a step with B = 0 it returns 0 and writes nothing.
 * Cost: about nx QP solves per instance (one factorisation per column). */
#define TMPC_JAC_OK 0          /* computed, strict complementarity holds                                                    */
#define TMPC_JAC_WEAK 1        /* computed, but a held row has |lam| < opts.lam_tresh or a row neither held nor relaxed has
                                  h(w*) < 10*opts.tol: the solution map has a kink there; J holds the active set as defined  */
#define TMPC_JAC_NOT_SOLVED 2  /* the step's status is not TMPC_OK: J is NaN                                                */
#define TMPC_JAC_SINGULAR 3    /* held rows dependent or reduced Hessian not positive definite: J is NaN                     */
int tmpc_feedback_jacobian(tmpc_handle* h, double* J, int32_t* jstatus, int dst_is_host, void* cuda_stream);

/* Vector-Jacobian product of the solution map (reverse mode of tmpc_feedback_jacobian), for B solutions:
 *     G_x0[b*nx + j] = sum_i V_u0[b*nu + i] du0_i/dx0_j + sum_e V_w[b*n_w + e] dw_e/dx0_j,
 * with the held set, the derivative and the jstatus values (TMPC_JAC_*) of tmpc_feedback_jacobian; G_x0 is NaN for statuses 2
 * and 3.  K = [H J_A'; J_A 0] is symmetric, so v' dw/dx0 is the init-row block mu of K [y; mu] = [v; 0]: ONE QP solve per
 * instance for both cotangents together, against nx for the Jacobian.
 * The solution: W (B*n_w), LAM (B*n_g), status (B) as a step returned them (W_dev, LAM_dev, status_dev of tmpc_step) and
 * `phase` = the phase that step used (its index mod p before the step, in [0, p)).  They are copied and linearised again in
 * buffers of the VJP, so a solution stored before later steps gives the same result as right after its step.  W == NULL selects
 * the last step's own solutions, status, phase and linearisation records; LAM and status must then be NULL and B equal that
 * step's batch size.  V_u0 (B*nu) and V_w (B*n_w) are the cotangents; either may be NULL, not both.
 * Buffers: all host memory if is_host != 0, else device memory on the handle's device (runs on `cuda_stream`).  Returns after its
 * kernels have finished.  Leaves the warm start, the phase index, the linearisation records, the QP step and multipliers, the
 * log, counters and timing unchanged.
 * API errors: the handle uses the Gauss-Newton Hessian (hessian_exact = 0 and not economic); a step is in flight; W == NULL and
 * no step has finished since tmpc_create / tmpc_reset; phase outside [0, p); both cotangents NULL.  B = 0 returns 0. */
int tmpc_solution_vjp(tmpc_handle* h, int64_t B, const double* W, const double* LAM, const int32_t* status, int32_t phase,
                      const double* V_u0, const double* V_w, double* G_x0, int32_t* jstatus, int is_host, void* cuda_stream);

/* plant = model integrator: Xn_dev[b] = F(X_dev[b], U_dev[b])   (closed_loop_tools.py:102) */
int tmpc_plant_step(tmpc_handle* h, const double* X_dev, const double* U_dev, int64_t B, double* Xn_dev,
                    void* cuda_stream);

/* plant Jacobian: JF_dev[b] = [dF/dx | dF/du] at (X_dev[b], U_dev[b]), nx x (nx+nu) row-major per instance, the first-order
 * sensitivities of the integrator of tmpc_plant_step (those of tmpc_stage_eval_host with order 1) */
int tmpc_plant_jacobian(tmpc_handle* h, const double* X_dev, const double* U_dev, int64_t B, double* JF_dev, void* cuda_stream);

/* closed-loop log of one (x,u) sample per instance: l_dev[b] = l(x_b,u_b) (economic stage cost of the model card),
 * h_dev[b*nh+i] = (C z_b + c)_i; either may be NULL   (closed_loop_tools.py:64-65, 98-99) */
int tmpc_stage_log(tmpc_handle* h, const double* X_dev, const double* U_dev, int64_t B, double* l_dev, double* h_dev,
                   void* cuda_stream);

/* per-step log of the last tmpc_step, copied into caller buffers of B elements each (any may be NULL); the buffers are
 * host memory if dst_is_host != 0, else device memory on the handle's device:
 * f objective, nAS active inequality rows, nACtot active-set changes vs the initial guess,
 * nAC stage-0 active-set changes vs the reference multipliers   (pmpc.py:815-856, sqp_method.py:203-219) */
int tmpc_get_log(tmpc_handle* h, double* f, int32_t* nAS, int32_t* nACtot, int32_t* nAC, int dst_is_host);
/* counters of the last tmpc_step: [0] SQP iterations summed over the batch, [1] kernel launches, [2] QP solves,
 * [3] stage linearisations (instance*stage), [4] plain dynamics evaluations (instance*stage) in the line search */
int tmpc_get_counters(const tmpc_handle* h, int64_t out[8]);
/* duration in ms of the last step's kernels by kind (CUDA events on the launch stream): [0] linearise, [1] qp,
 * [2] line search + convergence, [3] whole step */
int tmpc_get_timing(const tmpc_handle* h, double out_ms[4]);

/* host evaluation of the compiled model's one-interval map and derivatives (offline tuning only, not the solve
 * path): n stages, order 0/1/2 -> xf (n*nx), S (n*nx*nz), T (n*nx*nz*nz) */
int tmpc_stage_eval_host(int32_t n, const double* x, const double* u, int32_t order, double* xf, double* S,
                         double* T);

/* in-run FP64 FMA peak micro-benchmark on the handle's device: returns TFLOP/s (2 flops per DFMA) */
int tmpc_fp64_peak(tmpc_handle* h, double* tflops);

#ifdef __cplusplus
}
#endif
#endif
