/* nmpc_b200.h -- C-ABI of the B200-native batched NMPC solver (libnmpc_b200.so).
 *
 * Drop-in boundary (SURVEY.md section 8b): this library sits behind the one call the reference
 * makes on its hot path,
 *     solver = nlpsol('solver','ipopt', nlp_prob, opts)       AllScripts/centralized_six_robots_implementation.py:345-346
 *     sol    = solver(x0=, p=, lbx=, ubx=, lbg=, ubg=)        AllScripts/centralized_six_robots_implementation.py:432
 * for the NLP family those scripts build (multiple-shooting unicycle robots with pairwise
 * collision rows, :207-352; single robot: casadi_test.py:34-109), plus the two warm-start
 * helpers of the MPC loop (shift(), :160-169, and the X0 shift at :465) and the Euler plant of
 * casadi_test.py:17-26.
 *
 * Conventions
 *  - plain C, no torch types; every array is IEEE double unless stated, row-major [B, .].
 *  - decision vector  w = [X_0; ...; X_N; U_0; ...; U_{N-1}]  (n = 3Nr(N+1) + 2Nr N), CasADi's
 *    column-major reshape of the reference's X (ns x N+1) and U (nc x N)          (:240-245,339)
 *  - parameter  p = [x0bar (3Nr); xs (3Nr)]                                        (:419)
 *  - constraint rows g: N+1 blocks of [3Nr equality rows ; M = Nr(Nr-1)/2 distance rows]; block 0 =
 *    X_0 - x0bar and M constant rows (3.5); block k+1 = Euler defect of stage k and the squared
 *    distances on X_k, pairs in lexicographic order                               (:278,282-331)
 *  - multipliers in CasADi's sign convention (L = f + lam_g'g + lam_x'x).
 *  - functions whose names end in _host take HOST pointers (pageable or pinned: they are handed to
 *    cudaMemcpyAsync as they are, so only pinned buffers overlap with device work), copy them into a
 *    device staging area owned by the handle, and synchronise before returning; all others take DEVICE
 *    pointers, are asynchronous on `stream` and never allocate.
 *  - a handle belongs to the CUDA device that was current in nmpc_create; every later call must be made
 *    with the same device current (checked: NMPC_EINVAL otherwise).
 *  - return value: 0 on success, <0 on an API error (nmpc_last_error() has the text).
 *    Non-convergence is NOT an error: it is reported per instance in status[], and the last
 *    iterate is returned, as CasADi does by default (the reference never reads the status).
 */
#ifndef NMPC_B200_H
#define NMPC_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct nmpc_desc {
    int Nr;        /* robots          (reference variable m,  ...six...py:199)  1..10 on the CUDA path */
    int N;         /* horizon         (reference variable N,  :198)                                 */
    double T;      /* sampling period (:197)                                                        */
    double Q[3];   /* diag state weights   (1, 5, 0.1)   :252-259                                   */
    double R[2];   /* diag control weights (0.5, 0.05)   :261-266                                   */
} nmpc_desc;

/* Solver options: the ones the reference sets (:345) and the IPOPT defaults that shape the path. */
typedef struct nmpc_opts {
    double tol;                       /* 1e-8                                   */
    int    max_iter;                  /* 2000  (:345)                           */
    double acceptable_tol;            /* 1e-8  (:345)                           */
    int    acceptable_iter;           /* 15                                     */
    double acceptable_obj_change_tol; /* 1e-6  (:345)                           */
    double dual_inf_tol;              /* 1                                      */
    double constr_viol_tol;           /* 1e-4                                   */
    double compl_inf_tol;             /* 1e-4                                   */
    double mu_init;                   /* 0.1                                    */
    double kappa_mu;                  /* 0.2   mu_linear_decrease_factor        */
    double theta_mu;                  /* 1.5   mu_superlinear_decrease_power    */
    double barrier_tol_factor;        /* 10                                     */
    double tau_min;                   /* 0.99                                   */
    double bound_push;                /* 0.01  (and slack_bound_push)           */
    double bound_frac;                /* 0.01  (and slack_bound_frac)           */
    double bound_relax_factor;        /* 1e-8                                   */
    double bound_mult_init_val;       /* 1                                      */
    double constr_mult_init_max;      /* 1e3                                    */
    double kappa_sigma;               /* 1e10                                   */
    double kappa_d;                   /* 1e-5                                   */
    double nlp_scaling_max_gradient;  /* 100                                    */
    int    max_soc;                   /* 4                                      */
    int    max_resto_iter;            /* 100  bound on the restoration fallback */
} nmpc_opts;

enum { NMPC_SOLVED = 0, NMPC_ACCEPTABLE = 1, NMPC_MAX_ITER = 2, NMPC_INFEASIBLE = 3, NMPC_NUMERICAL = 4 };

/* stats[B][NMPC_NSTATS] */
enum { NMPC_ST_KKT_ERR = 0, NMPC_ST_PRIMAL_INF, NMPC_ST_DUAL_INF, NMPC_ST_COMPL, NMPC_ST_MU,
       NMPC_ST_N_REG, NMPC_ST_N_RESTO, NMPC_ST_N_SOC, NMPC_ST_N_FACTOR, NMPC_ST_N_LS,
       NMPC_ST_FILTER_EVICT,   /* filter entries dropped because the fixed-size filter was full (IPOPT's is unbounded): 0 on every parity case */
       NMPC_NSTATS };

enum { NMPC_EINVAL = -1, NMPC_EBOUNDS = -2, NMPC_ENOTSUP = -3, NMPC_ECUDA = -4, NMPC_ENOMEM = -5 };

typedef struct nmpc_handle nmpc_handle;

void nmpc_default_opts(nmpc_opts *o);
const char *nmpc_last_error(void);

/* Replaces the nlpsol(...) factory (:345-346).  The handle owns only immutable problem metadata. */
int nmpc_create(const nmpc_desc *d, const nmpc_opts *o, nmpc_handle **out);
void nmpc_destroy(nmpc_handle *h);

/* Launch tuning (no effect on results).  These used to be environment variables read inside nmpc_create; they are explicit
 * now so that nothing on the product path depends on the process environment.
 *   convoy            0 off, 1 the warps of a CTA meet at the start of every interior-point iteration, 2 (default) also
 *                     before the forward pass (instruction-cache locality of the one-warp-per-instance path)
 *   ctas_per_sm       > 0: cap on resident CTAs per SM (occupancy experiments); 0 = as many as fit
 *   force_block_path  != 0: run any Nr on the CTA-per-instance dense-block solver (test hook)
 *   thread_min_batch  > 0: batches at least this large of the one-robot static-obstacle family use the thread-per-instance
 *                     solver; 0 = never.  Ignored by nmpc_create_moving_obstacles and nmpc_create_tracking_obstacles (that
 *                     solver takes one static table) */
typedef struct nmpc_tuning { int convoy, ctas_per_sm, force_block_path, thread_min_batch; } nmpc_tuning;
void nmpc_default_tuning(nmpc_tuning *t);
/* nmpc_create / nmpc_create_obstacles (n_obs > 0) with explicit tuning; t == NULL means the defaults. */
int nmpc_create_tuned(const nmpc_desc *d, const nmpc_opts *o, const nmpc_tuning *t, int n_obs, const double *obs, nmpc_handle **out);

int nmpc_n(const nmpc_handle *h);        /* decision variables                         */
int nmpc_mg(const nmpc_handle *h);       /* constraint rows                            */
int nmpc_np(const nmpc_handle *h);       /* parameters (6 Nr, or 3 Nr + 5 Nr N tracking; + 3 N n_obs with obstacles in p) */
int nmpc_nnz_jac(const nmpc_handle *h);  /* 3Nr + N(11Nr+4M)   CasADi's CCS of dg/dw   */
int nmpc_nnz_hess(const nmpc_handle *h); /* N(6Nr+2M)          lower triangle          */

/* Bytes of device scratch nmpc_solve needs for a batch of B (independent of B beyond the
 * number of resident warps, so one workspace serves any batch size <= the B asked for). */
size_t nmpc_workspace_bytes(const nmpc_handle *h, int B);
/* Same when lbx/ubx/lbg/ubg are per-instance (bounds_batched = 1): adds B sets of stage-layout bound rows. */
size_t nmpc_workspace_bytes_batched_bounds(const nmpc_handle *h, int B);

/* Replaces  sol = solver(x0=,p=,lbx=,ubx=,lbg=,ubg=)  (:432) for B independent instances.
 * bounds_batched = 0: lbx/ubx [n], lbg/ubg [mg] shared by the batch; 1: [B,n] / [B,mg].
 * Outputs x [B,n], f [B], g [B,mg], lam_x [B,n], lam_g [B,mg], status/iters [B] (int32),
 * stats [B,NMPC_NSTATS]; any output except x may be NULL. */
int nmpc_solve(nmpc_handle *h, int B, const double *x0, const double *p,
               const double *lbx, const double *ubx, const double *lbg, const double *ubg,
               int bounds_batched, double *x, double *f, double *g, double *lam_x, double *lam_g,
               int32_t *status, int32_t *iters, double *stats,
               void *workspace, size_t workspace_bytes, void *stream);

/* Static circular obstacles (the reference's obstacle-avoidance scripts, first_/third_scenario_mpc_obstacle_avoidance.py:96-152):
 * same variables, cost and dynamics, plus n_obs rows per robot and stage
 *     sqrt((x_i - ox)^2 + (y_i - oy)^2) - clearance          on X_k, k = 0..N-1
 * with clearance = rob_dim + r_obs (:125), bounded below by the margin the scripts put in lbg (0.05 / 0.1) and above by +inf.
 * obs: HOST array [n_obs][3] = (ox, oy, clearance).  Row layout of g / lbg / ubg / lam_g (as the scripts build it, :109-125):
 * [X_0 - x0bar (3 Nr)], then for k = 0..N-1: [defect rows (3 Nr); pair rows (M, none for one robot); obstacle rows, robot-major
 * (Nr n_obs)]; mg = 3 Nr + N (3 Nr + M + Nr n_obs).  Runs on the warp-per-instance path for 1..4 robots while M + Nr n_obs <= 32
 * (one robot with up to 32 obstacles; the reference's scripts have one robot and 1, 4 or 6), else on the CTA-per-instance
 * dense-block path; nmpc_eval and the CCS patterns are not available for this family. */
int nmpc_create_obstacles(const nmpc_desc *d, const nmpc_opts *o, int n_obs, const double *obs, nmpc_handle **out);

/* Static-obstacle family with the obstacle geometry in p (per instance, per stage): scenario sweeps over obstacle layouts in one
 * batch, and obstacles that move along known or predicted trajectories over the horizon.
 *     p = [x0bar (3 Nr); xs (3 Nr); O],  O = [N][n_obs][3] = (ox, oy, clearance) of obstacle o at stage k = 0..N-1,
 *     nmpc_np = 6 Nr + 3 N n_obs.
 * Row (k, i, o), on X_k, is sqrt((x_{k,i} - ox_{k,o})^2 + (y_{k,i} - oy_{k,o})^2) - c_{k,o}.  Variables, g row layout, mg, bounds,
 * status and stats are those of nmpc_create_obstacles, and so is the path (warp-per-instance for 1..4 robots while
 * M + Nr n_obs <= 32, else the dense-block path; t->force_block_path is honoured, t->thread_min_batch is ignored).  A block O that
 * repeats one table at every stage gives bit for bit what nmpc_create_obstacles with that table gives.  The clearances are device
 * data and are NOT validated (a negative one is the caller's responsibility).  1 <= n_obs <= 32, else NMPC_EINVAL; t == NULL
 * means the default tuning.  nmpc_eval and the CCS patterns return NMPC_ENOTSUP; nmpc_shift and nmpc_plant work. */
int nmpc_create_moving_obstacles(const nmpc_desc *d, const nmpc_opts *o, const nmpc_tuning *t, int n_obs, nmpc_handle **out);

/* Trajectory tracking: the centralized family with a time-varying state AND control reference per instance and stage (e.g. the
 * output of a planner), instead of one goal xs.
 *     p = [x0bar (3 Nr); Z[0]; ...; Z[N-1]],  Z[k] = [xr_k (3 Nr); ur_k (2 Nr)] laid out like the stage vector z_k = [X_k; U_k],
 *     nmpc_np = 3 Nr + 5 Nr N,
 *     cost = sum_{k<N} (X_k - xr_k)' Q (X_k - xr_k) + (U_k - ur_k)' R (U_k - ur_k)   (no terminal term, no wrap of theta).
 * ur_k is the feed-forward control: with ur = 0, R pulls v and omega toward zero and the robot lags a moving reference.
 * Everything else is what nmpc_create gives: variables, g rows (with the dummy rows of block 0), mg, bounds, nnz_jac / nnz_hess
 * and the CCS patterns, status, stats, the path (warp-per-instance for 1..10 robots, dense blocks for 11..64;
 * t->force_block_path is honoured, t == NULL means the default tuning), nmpc_shift, nmpc_plant and nmpc_set_order.
 * Guarantee: if every Z[k] = [xs; 0], the outputs are bit for bit those of nmpc_create with p = [x0bar; xs].
 * nmpc_eval works on the handle with p [B, nmpc_np]: its gradient includes both references, its Jacobian and Hessian are
 * those of nmpc_create. */
int nmpc_create_tracking(const nmpc_desc *d, const nmpc_opts *o, const nmpc_tuning *t, nmpc_handle **out);

/* Trajectory tracking among obstacles: the moving-obstacle family (nmpc_create_moving_obstacles) with the per-stage reference of
 * nmpc_create_tracking in place of the goal xs, e.g. a planner's path with feed-forward controls, tracked while the collision and
 * obstacle rows stay hard constraints.
 *     p = [x0bar (3 Nr); Z[0]; ...; Z[N-1]; O],  Z[k] = [xr_k (3 Nr); ur_k (2 Nr)],  O = [N][n_obs][3] = (ox, oy, clearance),
 *     nmpc_np = 3 Nr + 5 Nr N + 3 N n_obs,
 *     cost = sum_{k<N} (X_k - xr_k)' Q (X_k - xr_k) + (U_k - ur_k)' R (U_k - ur_k).
 * Row (k, i, o), on X_k, is that of nmpc_create_moving_obstacles against table O[k].  Everything else is what
 * nmpc_create_moving_obstacles gives: variables, g row layout (no dummy rows in block 0), mg = 3 Nr + N (3 Nr + M + Nr n_obs),
 * bounds, status, stats and the path (warp-per-instance for 1..4 robots while M + Nr n_obs <= 32, else the dense-block path;
 * t->force_block_path is honoured, t->thread_min_batch is ignored, t == NULL means the default tuning).
 * Guarantee: if every Z[k] = [xs; 0], the outputs are bit for bit those of nmpc_create_moving_obstacles with p = [x0bar; xs; O].
 * 1 <= n_obs <= 32, else NMPC_EINVAL.  nmpc_eval and the CCS patterns return NMPC_ENOTSUP; nmpc_shift, nmpc_plant,
 * nmpc_set_order, nmpc_solve_host and nmpc_solve_trace work. */
int nmpc_create_tracking_obstacles(const nmpc_desc *d, const nmpc_opts *o, const nmpc_tuning *t, int n_obs, nmpc_handle **out);

/* Small generic optimal-control problems, one GPU thread per instance.  model NMPC_OCP_VAN_DER_POL is the direct-multiple-shooting
 * demo of mpc_pose_control_casadi.py:22-114: 2 states, 1 control, N intervals over the horizon T, each integrated by rk_steps RK4
 * steps together with the cost quadrature; decision vector INTERLEAVED [X_0, U_0, X_1, ..., U_{N-1}, X_N] (n = 3N + 2, :77-106),
 * g = F(X_k, U_k) - X_{k+1} (mg = 2N, :104), no parameter vector (pass p = NULL).  The initial state must be fixed through
 * lbx == ubx on X_0 (:79-80; IPOPT's make_parameter treatment); other variables must have lb < ub.  o == NULL: IPOPT defaults
 * (max_iter 3000).  nmpc_solve / nmpc_solve_host / nmpc_n / nmpc_mg work on the handle; shift, plant and eval do not apply. */
enum { NMPC_OCP_VAN_DER_POL = 1 };
int nmpc_create_ocp(int model, int N, double T, int rk_steps, const nmpc_opts *o, nmpc_handle **out);

/* Scheduling hint for the following nmpc_solve* calls on this handle: order [len] (DEVICE int32, caller owned, a permutation
 * of 0..len-1) is the sequence in which the persistent teams pull instances from the work queue; NULL (len ignored) restores
 * index order.  Instances differ in iteration count (17 on average, up to 70, one MPC step after a solve), so a closed loop
 * that passes the previous step's iteration counts sorted in descending order (longest first) shortens the tail of the launch.
 * Results do not depend on the order.  The array must stay valid, and its contents must be complete on the stream the solve
 * is launched on (nmpc_solve_host uses the handle's own stream: synchronise the producer first), until the hint is replaced.
 * A solve whose batch size differs from len fails with NMPC_EINVAL; entries outside 0..len-1 are skipped by the kernel
 * (the outputs of the instances a broken permutation leaves out are not written), so a stale or corrupt order can never
 * cause an out-of-bounds access. */
int nmpc_set_order(nmpc_handle *h, const int32_t *order, int len);

/* nmpc_solve plus a per-iteration trace [B][max_trace][8] = (mu, scaled KKT error, theta, f, alpha_primal,
 * alpha_dual, delta_w, line-search trials) -- the parity tests compare it with the oracle's trace. */
int nmpc_solve_trace(nmpc_handle *h, int B, const double *x0, const double *p,
                     const double *lbx, const double *ubx, const double *lbg, const double *ubg,
                     int bounds_batched, double *x, double *f, double *g, double *lam_x, double *lam_g,
                     int32_t *status, int32_t *iters, double *stats, double *trace, int max_trace,
                     void *workspace, size_t workspace_bytes, void *stream);

/* Parametric sensitivities of returned solutions: how x* moves when p moves (sIPOPT's sensitivity; CasADi's forward and reverse
 * derivatives of an nlpsol's x with respect to p).  Inputs are what nmpc_solve returned for B instances (x, lam_x [B,n],
 * lam_g [B,mg], DEVICE) with the p [B,np] and the bounds of that solve (bounds_batched as in nmpc_solve).  From them the call
 * rebuilds, per instance, the interior-point KKT matrix at the point, with CasADi's signs (L = f + lam_g'g + lam_x'x):
 *     K = [[W + Sx, J'], [J, -Ss^-1]],  W = Hessian of L,  Sx_i = |lam_x_i| / d_i,  Ss_j = |lam_g_j| / d_j on inequality rows,
 * d the distance of x_i (of g_j(x)) to the bound its multiplier pushes against, relaxed by bound_relax_factor (max(1,|b|)
 * scaled) as in the solve; no finite bound: 0; equality rows stay equalities, the constant block-0 rows get weight 0.  One
 * factorisation of K (the solve's stage-wise Riccati sweep, no regularisation) and one forward pass give
 *     nmpc_solution_vjp:  K [a; b] = [x_bar; 0],  p_bar = -(d2L/dx dp)' a - (dg/dp)' b          (reverse mode, [B,n] -> [B,np])
 *                         i.e. p_bar[x0bar] = b of the block-0 rows, p_bar[xs] = 2Q sum_{k<N} a[X_k];
 *                         tracking: p_bar[xr_k] = 2Q a[X_k], p_bar[ur_k] = 2R a[U_k]
 *     nmpc_solution_jvp:  K [x_dot; lam_dot] = -[d2L/dx dp p_dot; dg/dp p_dot]                  (forward mode, [B,np] -> [B,n])
 * At a strictly complementary KKT point this is the active-set implicit-function derivative of x* with respect to p up to O(1/S) on the active
 * bounds, i.e. about bound_relax_factor relative.  sens_status [B] (int32, may be NULL): 0 ok; 1 wrong inertia (a pivot <= 0:
 * second-order sufficiency fails at the point, the derivative is not defined) -- the instance's outputs are NaN; a negative
 * NMPC_E* code when the bounds are rejected as nmpc_solve rejects them (outputs NaN).  Handles from nmpc_create and
 * nmpc_create_tracking with 1..10 robots, whatever their tuning or solve path; the obstacle families, 11..64 robots and the
 * small-OCP family return NMPC_ENOTSUP.  NULL inputs, B <= 0, a handle created on another device or a workspace smaller than
 * nmpc_sensitivity_workspace_bytes(h, B, bounds_batched) return NMPC_EINVAL.  Asynchronous on stream; the handle's state
 * (including the nmpc_set_order hint, which does not apply) is left unchanged. */
int nmpc_solution_vjp(nmpc_handle *h, int B, const double *x, const double *lam_x, const double *lam_g, const double *p,
                      const double *lbx, const double *ubx, const double *lbg, const double *ubg, int bounds_batched,
                      const double *x_bar, double *p_bar, int32_t *sens_status, void *workspace, size_t workspace_bytes,
                      void *stream);
int nmpc_solution_jvp(nmpc_handle *h, int B, const double *x, const double *lam_x, const double *lam_g, const double *p,
                      const double *lbx, const double *ubx, const double *lbg, const double *ubg, int bounds_batched,
                      const double *p_dot, double *x_dot, int32_t *sens_status, void *workspace, size_t workspace_bytes,
                      void *stream);
/* Device scratch of both calls and of nmpc_solution_x0_jacobian (0 for an unsupported handle or B <= 0). */
size_t nmpc_sensitivity_workspace_bytes(const nmpc_handle *h, int B, int bounds_batched);

/* Advanced-step NMPC (asNMPC, Zavala & Biegler 2009): solve for a predicted initial state x0bar = p[0:3Nr] while the system
 * moves (preparation), then, once the state is measured, correct that solution to first order in one cheap launch (feedback).
 * nmpc_solution_x0_jacobian: jac [B][3Nr][n] (DEVICE), jac[b][j] = (dx* / dp) e_j, j < 3Nr -- exactly what
 *     nmpc_solution_jvp returns for that seed (same layout as x, X_0 rows = e_j).  One factorisation of K per instance and 3Nr
 *     forward passes; inputs, sens_status, workspace (nmpc_sensitivity_workspace_bytes), supported handles and error codes as
 *     nmpc_solution_jvp.
 * nmpc_advanced_step: x_corr [B,n] = x + sum_j jac[j] (x0bar_meas - p[0:3Nr])_j (x0bar_meas [B][3Nr], summed in order
 *     j = 0..3Nr-1); a variable with a finite bound is then clamped to [min(lbx_i, x_i), max(ubx_i, x_i)] (never pulled further
 *     outside a bound the solve left it just beyond); the X_0 rows are x0bar_meas exactly; an instance with sens_status != 0
 *     keeps x (X_0 = x0bar_meas).  Collision rows are not projected: the correction is first order, the next solve restores
 *     them.  lbx / ubx [n] or [B,n] (bounds_batched); all pointers DEVICE and non-NULL.  One launch, asynchronous on stream;
 *     supported handles and error codes as nmpc_solution_jvp (no workspace).
 * Both calls leave the handle's state unchanged. */
int nmpc_solution_x0_jacobian(nmpc_handle *h, int B, const double *x, const double *lam_x, const double *lam_g, const double *p,
                              const double *lbx, const double *ubx, const double *lbg, const double *ubg, int bounds_batched,
                              double *jac, int32_t *sens_status, void *workspace, size_t workspace_bytes, void *stream);
int nmpc_advanced_step(nmpc_handle *h, int B, const double *x, const double *jac, const int32_t *sens_status, const double *p,
                       const double *x0bar_meas, const double *lbx, const double *ubx, int bounds_batched, double *x_corr,
                       void *stream);

/* Distributed NMPC: S scenarios of R robots, each robot solved as its own one-robot instance (instance s R + r) against its
 * teammates' predicted paths, which this call exchanges on the device.  For a one-robot handle of nmpc_create_moving_obstacles or
 * nmpc_create_tracking_obstacles with K = n_obs, it writes into p [S R][nmpc_np] (row s R + a):
 *   - x0bar = state[s][a] (state [S][R][3], current poses);
 *   - the obstacle block O[N][K][3], at p + nmpc_np - 3 N K: O[k][o] = (x, y, clearance) of the o-th selected teammate's
 *     prediction at stage k.  Robot j's prediction is its pose at k = 0 and X_{min(k+1, N)} of its plan for k = 1..N-1 (plan
 *     [S R][n], the last solution in the handle's layout, X_k at 3k: the plan shifted by one period with the last stage
 *     repeated, as nmpc_shift does); plan == NULL (no plan yet) holds the pose at every stage.  Robot a's candidates are the
 *     other robots of its scenario, with key (d2, j), d2 = the smallest squared xy distance between the two predictions over
 *     k < N; the K smallest keys are selected in lexicographic order (ties go to the lower index), o in key order.  With
 *     R - 1 < K the remaining slots hold an inactive obstacle: the robot's own pose + (1e6, 0) at every stage, clearance 0;
 * nothing else (xs, or Z on a tracking handle) is touched: goals and references are the caller's.  min_dist [S R] (may be NULL)
 * gets the distance from each robot's pose to the nearest other robot of its scenario, over all R (+inf for R = 1).  Squares and
 * sums round to nearest without FMA contraction, the square root is correctly rounded, positions and the clearance are copied.
 * A row of robot a on stage 0 sits on the fixed X_0: a pair already closer than clearance + the obstacle rows' lbg margin makes
 * the instance infeasible, which the solve reports per instance (returning the last iterate) as for any other instance.
 * All pointers are DEVICE pointers; one launch (counted by nmpc_launch_count), asynchronous on stream, no allocation.  Other
 * handles: NMPC_ENOTSUP.  S <= 0, R <= 0, S R >= 2^31, NULL state or p, a clearance that is negative or not finite, or a
 * handle created on another device: NMPC_EINVAL. */
int nmpc_neighbour_obstacles(nmpc_handle *h, int S, int R, const double *state, const double *plan, double clearance,
                             double *p, double *min_dist, void *stream);

/* Same call with HOST buffers (what a CasADi-style caller has): H2D of the inputs, solve, D2H of
 * the requested outputs, synchronous.  Staging buffers live in the handle and grow on demand. */
int nmpc_solve_host(nmpc_handle *h, int B, const double *x0, const double *p,
                    const double *lbx, const double *ubx, const double *lbg, const double *ubg,
                    int bounds_batched, double *x, double *f, double *g, double *lam_x, double *lam_g,
                    int32_t *status, int32_t *iters, double *stats);

/* Warm-start shift between MPC steps: u0 = [u[1:]; u[-1]] (shift(), :160-169) and
 * X0 = [X[1:]; X[N-1]] (:465 -- the reference appends row N-1, not row N).  [B,n] -> [B,n]. */
int nmpc_shift(nmpc_handle *h, int B, const double *x_prev, double *x0_next, void *stream);

/* Euler plant of casadi_test.py:17-26: state <- state + T f(state, u), u = first control of x_opt
 * (x_opt [B,n]); state, state_next [B,3Nr] (may alias). */
int nmpc_plant(nmpc_handle *h, int B, const double *state, const double *x_opt, double *state_next,
               void *stream);

/* Stand-alone derivative evaluation (what CasADi's AD hands IPOPT, SURVEY.md a17): for B points
 * w [B,n], p [B,nmpc_np] (6 Nr; a tracking handle's 3 Nr + 5 Nr N), lam_g [B,mg]:  f [B], grad [B,n], g [B,mg], jac [B,nnz_jac] and
 * hess [B,nnz_hess] (CCS value order of nmpc_jac_pattern / nmpc_hess_pattern).  Outputs may be NULL. */
int nmpc_eval(nmpc_handle *h, int B, const double *w, const double *p, const double *lam_g,
              double *f, double *grad, double *g, double *jac, double *hess, void *stream);

/* CCS patterns (HOST int32 arrays: colptr [n+1], rowidx [nnz]). */
int nmpc_jac_pattern(const nmpc_handle *h, int32_t *colptr, int32_t *rowidx);
int nmpc_hess_pattern(const nmpc_handle *h, int32_t *colptr, int32_t *rowidx);

/* Measurement helper: sustained FP64 FMA throughput of the device (TFLOP/s) from a register-only DFMA
 * kernel -- the roofline denominator for the factorisation (MEASURED_PEAKS.json has no FP64 figure). */
int nmpc_probe_fp64(double *tflops_out);
/* Same for the FP64 tensor-core instruction (mma.sync.m8n8k4.f64, DMMA; tcgen05 has no f64 kind): the number behind the
 * dense-block path's choice of register tiles on the FP64 FMA pipe (csrc/block_solver.cuh). */
int nmpc_probe_dmma(double *tflops_out);

/* Debug aid: cycle counters of the phases of the dense-block factorisation (Nr > 10), CTA 0 only:
 * [0] stage-parallel pre-pass, [1] p + P r mat-vec, [2] stage-matrix assembly, [3] control-block elimination,
 * [4] first contraction, [5] second contraction.  reset != 0 clears the counters after the read. */
int nmpc_debug_block_profile(long long *out16, int reset);

/* Number of kernel launches issued by this handle so far (bench.py's gpu_launches). */
long long nmpc_launch_count(const nmpc_handle *h);

#ifdef __cplusplus
}
#endif
#endif
