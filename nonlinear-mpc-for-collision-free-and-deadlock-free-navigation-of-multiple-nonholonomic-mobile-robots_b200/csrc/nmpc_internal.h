/* Internal plain structs shared by the C-ABI (nmpc_b200.cu) and the kernels. */
#ifndef NMPC_INTERNAL_H
#define NMPC_INTERNAL_H
#include "nmpc_b200.h"

#define NMPC_LANES 32
#define NMPC_FILTER_CAP 256     /* filter entries per barrier subproblem (global scratch; overflow is counted in the stats) */
#define NMPC_FILTER_CAP_SMALL 64 /* the thread-per-instance small-OCP solver keeps its filter in local memory */
#define NMPC_DUMMY_ROW_VALUE 3.5 /* centralized_six_robots_implementation.py:278 */
#define NMPC_NTRACE 8
#define NMPC_MAX_ROBOTS 64
#define NMPC_MAX_OBSTACLES 32

/* Stage-layout bound rows prepared by prep_bounds_kernel, each [S][32] doubles per bound set:
 *   BL, BU : relaxed variable bounds of stage k (lanes 0..3Nr-1 states, 3Nr..5Nr-1 controls)
 *   CE     : right-hand side of the equality rows of block k (lanes < 3Nr)
 *   DL, DU : relaxed bounds of the inequality rows of block k (lanes < M)                     */
enum { NMPC_BR_BL = 0, NMPC_BR_BU, NMPC_BR_CE, NMPC_BR_DL, NMPC_BR_DU, NMPC_BR_COUNT };

typedef struct NmpcSolveParams {
    int Nr, N, B;
    double T, Q[3], R[2];
    nmpc_opts o;
    const double *x0, *p;            /* [B,n], [B,6Nr]                                  */
    const double *brows;             /* [nb][NMPC_BR_COUNT][S][32], nb = 1 or B          */
    long long bstride;               /* doubles between bound sets (0 when shared)       */
    const int *bound_err;            /* device flag written by prep_bounds_kernel        */
    double *x, *f, *g, *lam_x, *lam_g;
    int *status, *iters;
    double *stats;
    double *trace;                   /* optional [B][max_trace][NMPC_NTRACE]             */
    int max_trace;
    double *ws;                      /* per-warp-slot scratch                            */
    long long ws_stride;             /* doubles per warp slot                            */
    int *counter;                    /* work queue                                       */
    const int *pairs;                /* [M][2] pair table (dense-block path only)        */
    const int *order;                /* optional [B] processing order of the instances   */
    int convoy;                      /* warp path: the CTA's warps start every IPM iteration together */
    int nobs, family;                /* static obstacles per robot; row layout (0 / 1)   */
    const double *obs;               /* [nobs][3] centre x, y, clearance radius (device) */
    const double *lbx, *ubx, *lbg, *ubg;  /* flat bounds (small-OCP family reads them directly) */
    int bounds_batched, rk_steps, np;
    int obs_in_p;                    /* obstacle family: geometry from p ([N][nobs][3] after x0bar, xs), not from obs */
} NmpcSolveParams;

/* Inputs and outputs of nmpc_solution_vjp / nmpc_solution_jvp (sens_kernel).  A struct of its own, passed next to
 * NmpcSolveParams, so that the solve kernels' parameter block stays as it is. */
typedef struct NmpcSensParams {
    const double *x, *lam_x, *lam_g; /* a returned point [B,n], [B,n], [B,mg]             */
    const double *seed;              /* reverse: x_bar [B,n];  forward: p_dot [B,np]      */
    double *out;                     /* reverse: p_bar [B,np]; forward: x_dot [B,n]       */
    int *status;                     /* [B] or NULL: 0 ok, 1 wrong inertia, < 0 bounds rejected */
    int reverse;
} NmpcSensParams;

#endif
