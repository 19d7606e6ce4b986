// Thread-per-instance solver for small generic optimal-control problems (SURVEY.md 8f-4).
//
// The reference's mpc_pose_control_casadi.py:22-114 (BASELINE.json configs[0]) is CasADi's direct-multiple-shooting demo: the
// Van der Pol oscillator  x1' = (1 - x2^2) x1 - x2 + u,  x2' = x1,  running cost x1^2 + x2^2 + u^2, T = 10, N = 20 intervals, each
// integrated by 4 RK4 steps together with its cost quadrature (:45-59); decision vector INTERLEAVED [X_0, U_0, X_1, U_1, ..., X_N]
// (:77-106); the initial state is fixed through lbw = ubw (:79-80), x1 >= -0.25 (:98), |u| <= 1 (:88-89); g = F(X_k, U_k) - X_{k+1}
// (:104); one solver(x0=, lbx=, ubx=, lbg=, ubg=) call with IPOPT's defaults (:110-113).
//
// Same interior-point driver (ipm_driver.cuh) as the unicycle solvers; what differs is the stage: dense dynamics Jacobians and an
// exact Hessian of the Lagrangian THROUGH the RK4 integrator, obtained with second-order forward-mode AD (hyper-dual numbers over
// the nx + nu stage inputs) in place of CasADi's AD.  A stage is 3 variables, so one thread runs a whole instance (all matrices
// are 3 x 3 or smaller and live in registers / local memory); a batch is one thread per instance.  The model is a functor
// (VanDerPol below): another small OCP only needs its own f(x, u) -> (xdot, L).
#pragma once
#include "nmpc_internal.h"
#include "ipm_driver.cuh"
#include "solver_body.cuh"
#include "bounds_prep.cuh"

// value, gradient and symmetric Hessian w.r.t. NV inputs (packed upper triangle, row-major)
template <int NV>
struct Jet2 {
    static constexpr int NH = NV * (NV + 1) / 2;
    double v, g[NV], h[NH];
    static __host__ __device__ constexpr int hi(int i, int j) { return i * NV - i * (i - 1) / 2 + (j - i); }   // i <= j
    static __host__ __device__ Jet2 constant(double c)
    {
        Jet2 r; r.v = c;
        for (int i = 0; i < NV; i++) r.g[i] = 0.0;
        for (int i = 0; i < NH; i++) r.h[i] = 0.0;
        return r;
    }
    static __host__ __device__ Jet2 variable(double c, int k) { Jet2 r = constant(c); r.g[k] = 1.0; return r; }
};
template <int NV> __host__ __device__ inline Jet2<NV> operator+(const Jet2<NV> &a, const Jet2<NV> &b)
{
    Jet2<NV> r; r.v = a.v + b.v;
    for (int i = 0; i < NV; i++) r.g[i] = a.g[i] + b.g[i];
    for (int i = 0; i < Jet2<NV>::NH; i++) r.h[i] = a.h[i] + b.h[i];
    return r;
}
template <int NV> __host__ __device__ inline Jet2<NV> operator-(const Jet2<NV> &a, const Jet2<NV> &b)
{
    Jet2<NV> r; r.v = a.v - b.v;
    for (int i = 0; i < NV; i++) r.g[i] = a.g[i] - b.g[i];
    for (int i = 0; i < Jet2<NV>::NH; i++) r.h[i] = a.h[i] - b.h[i];
    return r;
}
template <int NV> __host__ __device__ inline Jet2<NV> operator*(double c, const Jet2<NV> &a)
{
    Jet2<NV> r; r.v = c * a.v;
    for (int i = 0; i < NV; i++) r.g[i] = c * a.g[i];
    for (int i = 0; i < Jet2<NV>::NH; i++) r.h[i] = c * a.h[i];
    return r;
}
template <int NV> __host__ __device__ inline Jet2<NV> operator*(const Jet2<NV> &a, const Jet2<NV> &b)
{
    Jet2<NV> r; r.v = a.v * b.v;
    for (int i = 0; i < NV; i++) r.g[i] = a.g[i] * b.v + a.v * b.g[i];
    for (int i = 0; i < NV; i++)
        for (int j = i; j < NV; j++)
            r.h[Jet2<NV>::hi(i, j)] = a.h[Jet2<NV>::hi(i, j)] * b.v + a.v * b.h[Jet2<NV>::hi(i, j)] + a.g[i] * b.g[j] + a.g[j] * b.g[i];
    return r;
}

// sin, cos, sqrt of a jet (chain rule to second order)
template <int NV> __host__ __device__ inline Jet2<NV> jet_unary(const Jet2<NV> &a, double f0, double f1, double f2)
{
    Jet2<NV> r; r.v = f0;
    for (int i = 0; i < NV; i++) r.g[i] = f1 * a.g[i];
    for (int i = 0; i < NV; i++)
        for (int j = i; j < NV; j++) r.h[Jet2<NV>::hi(i, j)] = f1 * a.h[Jet2<NV>::hi(i, j)] + f2 * a.g[i] * a.g[j];
    return r;
}
template <int NV> __host__ __device__ inline Jet2<NV> jsin(const Jet2<NV> &a) { double s, c; sincos(a.v, &s, &c); return jet_unary(a, s, c, -s); }
template <int NV> __host__ __device__ inline Jet2<NV> jcos(const Jet2<NV> &a) { double s, c; sincos(a.v, &s, &c); return jet_unary(a, c, -s, -c); }
template <int NV> __host__ __device__ inline Jet2<NV> jsqrt(const Jet2<NV> &a) { const double r = sqrt(a.v); return jet_unary(a, r, 0.5 / r, -0.25 / (r * a.v)); }

// what a model needs to know about the instance
struct OcpCtx {
    int N, rk_steps, nobs;
    double T, Q[3], R[2];
    const double *p;     // this instance's parameter vector (may be NULL)
    const double *obs;   // [nobs][3]
};

// mpc_pose_control_casadi.py:25-35, 45-59, 77-106
struct VanDerPol {
    static constexpr int NX = 2, NU = 1, MAXI = 0;
    static constexpr bool INIT_ROWS = false;      // the initial state is fixed through its bounds (:79-80)
    static constexpr int EQ_SIGN = 1;             // shooting rows are reported as F(X_k, U_k) - X_{k+1} (:104)
    template <class S> static __host__ __device__ void f(const S *x, const S *u, S *xdot, S &L)
    {
        const S one = S::constant(1.0);
        xdot[0] = (one - x[1] * x[1]) * x[0] - x[1] + u[0];
        xdot[1] = x[0];
        L = x[0] * x[0] + x[1] * x[1] + u[0] * u[0];
    }
    template <class S> static __device__ void step(const OcpCtx &c, int, const S *x, const S *u, S *xf, S &q);
    static __device__ int n_ineq(const OcpCtx &) { return 0; }
    template <class S> static __device__ S ineq(const OcpCtx &, int, const S *) { return S::constant(0.0); }
    static NMPC_HD long long n(int N, int) { return 3LL * N + 2; }
    static NMPC_HD long long mg(int N, int) { return 2LL * N; }
    static __device__ long long xidx(const OcpCtx &, int k, int l) { return 3LL * k + l; }                 // interleaved (:77-106)
    static __device__ long long grow_eq(const OcpCtx &, int k, int i) { return 2LL * (k - 1) + i; }        // F(z_{k-1}) - X_k, k >= 1
    static __device__ long long grow_in(const OcpCtx &, int, int) { return -1; }
    static __device__ double x0bar(const OcpCtx &, int) { return 0.0; }
};

// first_scenario_mpc_obstacle_avoidance.py:75-152: one unicycle, Euler shooting, quadratic tracking cost, static circular obstacles
struct UnicycleObstacles {
    static constexpr int NX = 3, NU = 2, MAXI = NMPC_MAX_OBSTACLES;
    static constexpr bool INIT_ROWS = true;       // g starts with X_0 - x0bar (:109)
    static constexpr int EQ_SIGN = -1;            // shooting rows are reported as X_{k+1} - (X_k + T f) (:122-123)
    template <class S> static __device__ void step(const OcpCtx &c, int, const S *x, const S *u, S *xf, S &q)
    {
        const S cs = jcos(x[2]), sn = jsin(x[2]);
        xf[0] = x[0] + c.T * (u[0] * cs); xf[1] = x[1] + c.T * (u[0] * sn); xf[2] = x[2] + c.T * u[1];     // :118-122
        q = S::constant(0.0);
        for (int i = 0; i < 3; i++) { const S e = x[i] - S::constant(c.p[3 + i]); q = q + c.Q[i] * (e * e); }   // :115
        for (int i = 0; i < 2; i++) q = q + c.R[i] * (u[i] * u[i]);
    }
    static __device__ int n_ineq(const OcpCtx &c) { return c.nobs; }
    template <class S> static __device__ S ineq(const OcpCtx &c, int i, const S *x)                        // :125
    {
        const S dx = x[0] - S::constant(c.obs[3 * i]), dy = x[1] - S::constant(c.obs[3 * i + 1]);
        return jsqrt(dx * dx + dy * dy) - S::constant(c.obs[3 * i + 2]);
    }
    static NMPC_HD long long n(int N, int) { return 3LL * (N + 1) + 2LL * N; }
    static NMPC_HD long long mg(int N, int nobs) { return 3 + (long long)N * (3 + nobs); }
    static __device__ long long xidx(const OcpCtx &c, int k, int l) { return l < 3 ? 3LL * k + l : 3LL * (c.N + 1) + 2LL * k + (l - 3); }
    static __device__ long long grow_eq(const OcpCtx &c, int k, int i) { return k == 0 ? i : 3 + (long long)(k - 1) * (3 + c.nobs) + i; }
    static __device__ long long grow_in(const OcpCtx &c, int k, int i) { return 3 + (long long)k * (3 + c.nobs) + 3 + i; }   // row on X_k, k < N
    static __device__ double x0bar(const OcpCtx &c, int i) { return c.p[i]; }
};

// one shooting interval: M fixed RK4 steps of size DT on the state and the cost quadrature (:45-59)
template <class Model, class S>
__host__ __device__ inline void rk4_interval(const S *x0, const S *u, int M, double DT, S *xf, S &qf)
{
    constexpr int NX = Model::NX;
    S X[NX], k1[NX], k2[NX], k3[NX], k4[NX], t[NX], q1, q2, q3, q4;
    for (int i = 0; i < NX; i++) X[i] = x0[i];
    qf = S::constant(0.0);
    for (int j = 0; j < M; j++) {
        Model::f(X, u, k1, q1);
        for (int i = 0; i < NX; i++) t[i] = X[i] + (DT / 2) * k1[i];
        Model::f(t, u, k2, q2);
        for (int i = 0; i < NX; i++) t[i] = X[i] + (DT / 2) * k2[i];
        Model::f(t, u, k3, q3);
        for (int i = 0; i < NX; i++) t[i] = X[i] + DT * k3[i];
        Model::f(t, u, k4, q4);
        for (int i = 0; i < NX; i++) X[i] = X[i] + (DT / 6) * (k1[i] + 2.0 * k2[i] + 2.0 * k3[i] + k4[i]);
        qf = qf + (DT / 6) * (q1 + 2.0 * q2 + 2.0 * q3 + q4);
    }
    for (int i = 0; i < NX; i++) xf[i] = X[i];
}

template <class S> __device__ void VanDerPol::step(const OcpCtx &c, int, const S *x, const S *u, S *xf, S &q)
{
    rk4_interval<VanDerPol, S>(x, u, c.rk_steps, c.T / c.N / c.rk_steps, xf, q);
}

template <class Model>
struct ThreadSolver {
    static constexpr int NX = Model::NX, NU = Model::NU, NZ = NX + NU, MAXI = Model::MAXI;
    static constexpr int LD = MAXI > 8 ? MAXI : 8;   // row length: stage variables (NZ <= 8) or inequality rows of a stage
    static constexpr bool INIT_ROWS = Model::INIT_ROWS;
    static_assert(NZ <= 8, "stage vector must fit the row");
    typedef Jet2<NZ> J2;
    static constexpr int NXH = NX * (NX + 1) / 2;
    typedef WarpSolver<1> WS;
    enum Row {
        R_Z, R_ZL, R_ZU, R_BL, R_BU, R_DZ, R_DZ2, R_GX, R_YC, R_YTC, R_YTC2, R_RC, R_CSOC, R_CE, R_LIN, R_DGV, R_ZT,
        R_S, R_VL, R_VU, R_DL, R_DU, R_YD, R_DS, R_DS2, R_YTD, R_YTD2, R_DSOC, R_GS, R_DQ, R_RD, R_ST, R_HV,
        R_COUNT
    };
    struct EvalOut { double pinf, viol, dinf, c0, cmu, ysum, zsum, theta, f, slog, sdamp; };
    struct StepInfo { double ap, az, gbd, tiny; };
    // per-stage cache of the discretised model (doubles per stage); inequality row i: value, gradient and Hessian w.r.t. X_k
    enum { C_F = 0, C_J = C_F + NX, C_HF = C_J + NX * NZ, C_Q = C_HF + NX * J2::NH, C_GQ = C_Q + 1, C_HQ = C_GQ + NZ,
           C_P = C_HQ + J2::NH, C_K = C_P + NX * NX, C_KF = C_K + NU * NX, C_H = C_KF + NU, C_I = C_H + J2::NH,
           CI_STRIDE = 1 + NX + NXH, C_COUNT = C_I + MAXI * CI_STRIDE };

    const NmpcSolveParams &P;
    OcpCtx ctx;
    double *ws, *cache;
    int N, S, inst, fn, ni;
    bool fixed0;
    double df, ny_nzb, nzb_cnt;
    int n_reg, n_resto, n_soc, n_fact, n_ls, n_evict;
    double fth[NMPC_FILTER_CAP_SMALL], fph[NMPC_FILTER_CAP_SMALL];

    static NMPC_HD long long ws_doubles(int N) { return (long long)(R_COUNT * LD + C_COUNT) * (N + 1); }

    __device__ ThreadSolver(const NmpcSolveParams &p, double *wsp) : P(p), ws(wsp) {}
    static __device__ __forceinline__ void tsync() {}
    __device__ __forceinline__ bool is_lead() const { return true; }
    __device__ __forceinline__ void iter_sync() const {}
    __device__ __forceinline__ void mid_sync() const {}
    __device__ __forceinline__ double *row(int r, int k) const { return ws + ((long long)r * S + k) * LD; }
    __device__ __forceinline__ double *cst(int k) const { return cache + (long long)k * C_COUNT; }
    __device__ __forceinline__ double *cin(int k, int i) const { return cst(k) + C_I + i * CI_STRIDE; }
    // variable l of stage k takes part in the optimisation (a fixed initial state and U_N do not)
    __device__ __forceinline__ bool valid(int k, int l) const { return l < (k < N ? NZ : NX) && !(fixed0 && k == 0 && l < NX); }
    __device__ __forceinline__ int kfirst() const { return INIT_ROWS ? 0 : 1; }   // first stage that carries equality rows
    static __device__ __forceinline__ int xh(int a, int b) { return a <= b ? a * NX - a * (a - 1) / 2 + (b - a) : xh(b, a); }

    __device__ void setup(int instance)
    {
        inst = instance; N = P.N; S = N + 1;
        ctx.N = N; ctx.T = P.T; ctx.rk_steps = P.rk_steps; ctx.nobs = P.nobs; ctx.obs = P.obs;
        ctx.p = P.p ? P.p + (long long)inst * P.np : nullptr;
        for (int i = 0; i < 3; i++) ctx.Q[i] = P.Q[i];
        for (int i = 0; i < 2; i++) ctx.R[i] = P.R[i];
        ni = Model::n_ineq(ctx);
        cache = ws + (long long)R_COUNT * LD * S;
        df = 1.0; fn = 0; fixed0 = false;
        n_reg = n_resto = n_soc = n_fact = n_ls = n_evict = 0;
    }
    __device__ bool bounds_rejected()
    {
        // A fixed INITIAL STATE (lbx == ubx on X_0) becomes a parameter, as IPOPT's default fixed_variable_treatment does;
        // any other fixed variable, lb > ub, a non-equality shooting row or an equality inequality-row is rejected.
        const long long n = Model::n(N, ctx.nobs), mg = Model::mg(N, ctx.nobs);
        const double *lb = P.lbx + (P.bounds_batched ? inst * n : 0), *ub = P.ubx + (P.bounds_batched ? inst * n : 0);
        const double *lg = P.lbg + (P.bounds_batched ? inst * mg : 0), *ug = P.ubg + (P.bounds_batched ? inst * mg : 0);
        int nfix0 = 0;
        for (int l = 0; l < NX; l++) nfix0 += lb[Model::xidx(ctx, 0, l)] == ub[Model::xidx(ctx, 0, l)];
        fixed0 = nfix0 == NX;
        int err = 0;
        if (INIT_ROWS ? nfix0 != 0 : !fixed0) err = NMPC_ENOTSUP;   // the initial state comes from the rows, or from the bounds, not both
        for (int k = 0; k <= N; k++) {
            for (int l = 0; l < LD; l++) {
                double blo = -NMPC_INF, bhi = NMPC_INF;
                if (l < (k < N ? NZ : NX)) {
                    const double lo = lb[Model::xidx(ctx, k, l)], hi = ub[Model::xidx(ctx, k, l)];
                    if (!(lo <= hi)) err = err ? err : NMPC_EBOUNDS;
                    else if (lo == hi && !(fixed0 && k == 0 && l < NX)) err = err ? err : NMPC_ENOTSUP;
                    if (!(fixed0 && k == 0 && l < NX)) { blo = nmpc_relax_lo(lo, P.o.bound_relax_factor); bhi = nmpc_relax_hi(hi, P.o.bound_relax_factor); }
                }
                row(R_BL, k)[l] = blo; row(R_BU, k)[l] = bhi;
                double ce = 0.0;
                if (l < NX && k >= kfirst()) {
                    const long long r = Model::grow_eq(ctx, k, l);
                    if (!(lg[r] == ug[r]) || !(lg[r] > -NMPC_INF && lg[r] < NMPC_INF)) err = err ? err : NMPC_ENOTSUP;
                    ce = lg[r];
                }
                row(R_CE, k)[l] = ce;
                double dl = -NMPC_INF, du = NMPC_INF;
                if (l < ni && k < N) {
                    const long long r = Model::grow_in(ctx, k, l);
                    dl = lg[r]; du = ug[r];
                    if (!(dl <= du)) err = err ? err : NMPC_EBOUNDS;
                    else if (dl == du) err = err ? err : NMPC_ENOTSUP;
                    dl = nmpc_relax_lo(dl, P.o.bound_relax_factor); du = nmpc_relax_hi(du, P.o.bound_relax_factor);
                }
                row(R_DL, k)[l] = dl; row(R_DU, k)[l] = du;
            }
        }
        if (err) {
            if (P.status) P.status[inst] = err;
            if (P.iters) P.iters[inst] = 0;
            return true;
        }
        return false;
    }

    // discretised model of stage k at the stage vector z: values, Jacobian, Hessians, inequality rows (into the stage cache)
    __device__ void model(int k, const double *z)
    {
        J2 x[NX], u[NU], xf[NX], qf;
        for (int i = 0; i < NX; i++) x[i] = J2::variable(z[i], i);
        for (int i = 0; i < NU; i++) u[i] = J2::variable(z[NX + i], NX + i);
        Model::template step<J2>(ctx, k, x, u, xf, qf);
        double *c = cst(k);
        for (int i = 0; i < NX; i++) {
            c[C_F + i] = xf[i].v;
            for (int l = 0; l < NZ; l++) c[C_J + i * NZ + l] = xf[i].g[l];
            for (int e = 0; e < J2::NH; e++) c[C_HF + i * J2::NH + e] = xf[i].h[e];
        }
        c[C_Q] = qf.v;
        for (int l = 0; l < NZ; l++) c[C_GQ + l] = qf.g[l];
        for (int e = 0; e < J2::NH; e++) c[C_HQ + e] = qf.h[e];
        for (int i = 0; i < ni; i++) {
            const J2 h = Model::template ineq<J2>(ctx, i, x);
            double *ci = cin(k, i);
            ci[0] = h.v;
            for (int a = 0; a < NX; a++) ci[1 + a] = h.g[a];
            for (int a = 0; a < NX; a++) for (int b = a; b < NX; b++) ci[1 + NX + xh(a, b)] = h.h[J2::hi(a, b)];
        }
    }
    __device__ __forceinline__ bool qact(int k, int i) const { return row(R_DL, k)[i] > -NMPC_INF || row(R_DU, k)[i] < NMPC_INF; }
    // equality residual of stage k: F(z_{k-1}) - X_k - ce (k >= 1), x0bar - X_0 - ce (k = 0, INIT_ROWS)
    __device__ __forceinline__ double eqres(int k, int i, const double *xk) const
    {
        return (k == 0 ? Model::x0bar(ctx, i) : cst(k - 1)[C_F + i]) - xk[i] - (k == 0 ? -1.0 : (double)Model::EQ_SIGN) * row(R_CE, k)[i];
    }

    __device__ __noinline__ void init_point()
    {
        const long long n = Model::n(N, ctx.nobs);
        const double *x0 = P.x0 + inst * n;
        const nmpc_opts &o = P.o;
        const double *lb = P.lbx + (P.bounds_batched ? inst * n : 0);
        double gmax = 0.0, cnt_z = 0.0, cnt_y = 0.0;
        for (int k = 0; k <= N; k++)
            for (int l = 0; l < LD; l++) {
                double z = (l < (k < N ? NZ : NX)) ? x0[Model::xidx(ctx, k, l)] : 0.0;
                if (fixed0 && k == 0 && l < NX) z = lb[Model::xidx(ctx, 0, l)];
                double zl = 0.0, zu = 0.0;
                if (valid(k, l)) {
                    const double lo = row(R_BL, k)[l], hi = row(R_BU, k)[l];
                    z = WS::push_in(z, lo, hi, o.bound_push, o.bound_frac);
                    if (lo > -NMPC_INF) { zl = o.bound_mult_init_val; cnt_z += 1.0; }
                    if (hi < NMPC_INF) { zu = o.bound_mult_init_val; cnt_z += 1.0; }
                }
                row(R_Z, k)[l] = z; row(R_ZL, k)[l] = zl; row(R_ZU, k)[l] = zu;
                row(R_YC, k)[l] = 0.0; row(R_CSOC, k)[l] = 0.0; row(R_YD, k)[l] = 0.0; row(R_DSOC, k)[l] = 0.0;
                row(R_S, k)[l] = 0.0; row(R_VL, k)[l] = 0.0; row(R_VU, k)[l] = 0.0;
            }
        for (int k = 0; k < N; k++) {   // objective scaling from the gradient at the starting point; slacks from the rows
            model(k, row(R_Z, k));
            for (int l = 0; l < NZ; l++)
                if (valid(k, l)) gmax = fmax(gmax, fabs(cst(k)[C_GQ + l]));
            for (int i = 0; i < ni; i++) {
                if (!qact(k, i)) continue;
                const double lo = row(R_DL, k)[i], hi = row(R_DU, k)[i];
                row(R_S, k)[i] = WS::push_in(cin(k, i)[0], lo, hi, o.bound_push, o.bound_frac);
                if (lo > -NMPC_INF) { row(R_VL, k)[i] = o.bound_mult_init_val; cnt_z += 1.0; }
                if (hi < NMPC_INF) { row(R_VU, k)[i] = o.bound_mult_init_val; cnt_z += 1.0; }
                cnt_y += 1.0;
            }
        }
        df = gmax > o.nlp_scaling_max_gradient ? fmax(o.nlp_scaling_max_gradient / gmax, 1e-8) : 1.0;
        nzb_cnt = cnt_z; ny_nzb = (double)(NX * (N + (INIT_ROWS ? 1 : 0))) + cnt_y + cnt_z;
    }

    __device__ __noinline__ void eval(bool full, double mu, double alpha, int rdz, int rds, bool trial, bool socacc, double asoc, EvalOut &E)
    {
        const double kd = P.o.kappa_d;
        const int rz = trial ? R_ZT : R_Z, rs = trial ? R_ST : R_S;
        if (trial)
            for (int k = 0; k <= N; k++)
                for (int l = 0; l < LD; l++) {
                    row(R_ZT, k)[l] = row(R_Z, k)[l] + (valid(k, l) ? alpha * row(rdz, k)[l] : 0.0);
                    row(R_ST, k)[l] = row(R_S, k)[l] + ((l < ni && k < N) ? alpha * row(rds, k)[l] : 0.0);
                }
        double pinf = 0, viol = 0, dinf = 0, c0 = 0, cmu = 0, ysum = 0, zsum = 0, th = 0, fo = 0, sdamp = 0, slog = 0;
        for (int k = 0; k < N; k++) model(k, row(rz, k));
        for (int k = kfirst(); k <= N; k++)   // equality rows
            for (int i = 0; i < NX; i++) {
                const double c = eqres(k, i, row(rz, k));
                pinf = fmax(pinf, fabs(c)); th += fabs(c); viol = fmax(viol, fabs(c));
                if (socacc) row(R_CSOC, k)[i] = asoc * row(R_CSOC, k)[i] + c;
                if (full) ysum += fabs(row(R_YC, k)[i]);
            }
        for (int k = 0; k < N; k++) {
            fo += cst(k)[C_Q];
            for (int i = 0; i < ni; i++) {   // inequality rows on X_k
                if (!qact(k, i)) continue;
                const double lo = row(R_DL, k)[i], hi = row(R_DU, k)[i], dv = cin(k, i)[0], s = row(rs, k)[i], dms = dv - s;
                const bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
                pinf = fmax(pinf, fabs(dms)); th += fabs(dms); viol = fmax(viol, fmax(lo - dv, dv - hi));
                if (socacc) row(R_DSOC, k)[i] = asoc * row(R_DSOC, k)[i] + dms;
                if (hl) slog += log(s - lo);
                if (hu) slog += log(hi - s);
                if (hl && !hu) sdamp += s - lo;
                if (hu && !hl) sdamp += hi - s;
                if (full) {
                    const double yd = row(R_YD, k)[i], vl = row(R_VL, k)[i], vu = row(R_VU, k)[i];
                    ysum += fabs(yd);
                    double t = -yd - vl + vu;
                    if (hl && !hu) t += kd * mu;
                    if (hu && !hl) t -= kd * mu;
                    dinf = fmax(dinf, fabs(t));
                    if (hl) { const double u = (s - lo) * vl; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(vl); }
                    if (hu) { const double u = (hi - s) * vu; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(vu); }
                }
            }
        }
        for (int k = 0; k <= N; k++)
            for (int l = 0; l < NZ; l++) {
                if (!valid(k, l)) continue;
                const double zk = row(rz, k)[l], lo = row(R_BL, k)[l], hi = row(R_BU, k)[l];
                const bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
                if (hl) slog += log(zk - lo);
                if (hu) slog += log(hi - zk);
                if (hl && !hu) sdamp += zk - lo;
                if (hu && !hl) sdamp += hi - zk;
                if (full) {
                    const double zl = row(R_ZL, k)[l], zu = row(R_ZU, k)[l];
                    double r = -zl + zu;
                    if (hl && !hu) r += kd * mu;
                    if (hu && !hl) r -= kd * mu;
                    if (k < N) {
                        r += df * cst(k)[C_GQ + l];
                        for (int i = 0; i < NX; i++) r += cst(k)[C_J + i * NZ + l] * row(R_YC, k + 1)[i];
                        if (l < NX) for (int i = 0; i < ni; i++) r += cin(k, i)[1 + l] * row(R_YD, k)[i];
                    }
                    if (l < NX && k >= kfirst()) r -= row(R_YC, k)[l];
                    dinf = fmax(dinf, fabs(r));
                    if (hl) { const double u = (zk - lo) * zl; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(zl); }
                    if (hu) { const double u = (hi - zk) * zu; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(zu); }
                }
            }
        E.pinf = pinf; E.viol = viol; E.theta = th; E.f = fo; E.slog = slog; E.sdamp = sdamp;
        if (full) { E.dinf = dinf; E.c0 = c0; E.cmu = cmu; E.ysum = ysum; E.zsum = zsum; }
    }

    __device__ bool factor_m(int mode, double mu, double delta, bool soc) { return factor(mode, mu, delta, soc); }
    // backward Riccati sweep with dense NZ x NZ stage matrices; false = a control pivot <= 0 (wrong inertia)
    __device__ __noinline__ bool factor(int mode, double mu, double delta, bool soc)
    {
        const double zeta = mode == 2 ? sqrt(mu) : 0.0, kd = P.o.kappa_d;
        n_fact++;
        for (int k = 0; k < N; k++) model(k, row(R_Z, k));
        for (int k = 0; k <= N; k++) {
            for (int l = 0; l < LD; l++) {
                double sig = 0.0, gx = 0.0, dg = 0.0;
                if (valid(k, l)) {
                    const double g0 = k < N ? df * cst(k)[C_GQ + l] : 0.0;
                    BlockSolver::sig_g(mode, kd, row(R_Z, k)[l], row(R_BL, k)[l], row(R_BU, k)[l], row(R_ZL, k)[l], row(R_ZU, k)[l], mu, g0, sig, gx);
                    dg = sig + delta + zeta;
                }
                row(R_GX, k)[l] = gx; row(R_HV, k)[l] = gx; row(R_DGV, k)[l] = dg;   // R_HV: stage gradient of the Riccati sweep
                if (l < NX) row(R_RC, k)[l] = (mode == 1 || k < kfirst()) ? 0.0 : (soc ? row(R_CSOC, k)[l] : eqres(k, l, row(R_Z, k)));
            }
            if (k < N) {
                double *c = cst(k);
                for (int e = 0; e < J2::NH; e++) {   // Hessian of the Lagrangian of stage k (exact, through the integrator)
                    double h = 0.0;
                    if (mode == 0) {
                        h = df * c[C_HQ + e];
                        for (int i = 0; i < NX; i++) h += row(R_YC, k + 1)[i] * c[C_HF + i * J2::NH + e];
                    }
                    c[C_H + e] = h;
                }
                for (int i = 0; i < ni; i++) {   // condensed inequality rows: slack and multiplier eliminated
                    double gs = 0.0, Dq = 0.0, rd = 0.0;
                    if (qact(k, i)) {
                        const double s = row(R_S, k)[i];
                        double sigs;
                        BlockSolver::sig_g(mode, kd, s, row(R_DL, k)[i], row(R_DU, k)[i], row(R_VL, k)[i], row(R_VU, k)[i], mu, 0.0, sigs, gs);
                        rd = mode == 1 ? 0.0 : (soc ? row(R_DSOC, k)[i] : cin(k, i)[0] - s);
                        Dq = sigs + delta;
                        const double hq = Dq * rd + gs, yq = mode == 0 ? row(R_YD, k)[i] : 0.0;
                        const double *ci = cin(k, i);
                        for (int a = 0; a < NX; a++) {
                            for (int b = a; b < NX; b++) c[C_H + J2::hi(a, b)] += Dq * ci[1 + a] * ci[1 + b] + yq * ci[1 + NX + xh(a, b)];
                            row(R_HV, k)[a] += ci[1 + a] * hq;
                        }
                    }
                    row(R_GS, k)[i] = gs; row(R_DQ, k)[i] = Dq; row(R_RD, k)[i] = rd;
                }
            }
        }
        double Pn[NX][NX], pn[NX];
        for (int i = 0; i < NX; i++) {
            for (int j = 0; j < NX; j++) Pn[i][j] = i == j ? row(R_DGV, N)[i] : 0.0;
            pn[i] = row(R_HV, N)[i];
            row(R_LIN, N)[i] = pn[i];
            for (int j = 0; j < NX; j++) cst(N)[C_P + i * NX + j] = Pn[i][j];
        }
        for (int k = N - 1; k >= 0; k--) {
            const double *c = cst(k);
            double AB[NX][NZ], Mm[NZ][NZ], mv[NZ], pr[NX], W[NX][NZ];
            for (int i = 0; i < NX; i++) for (int l = 0; l < NZ; l++) AB[i][l] = c[C_J + i * NZ + l];
            for (int i = 0; i < NX; i++) {   // dx_{k+1} = A dx + B du + rc_{k+1}
                double a = pn[i];
                for (int j = 0; j < NX; j++) a += Pn[i][j] * row(R_RC, k + 1)[j];
                pr[i] = a;
            }
            for (int i = 0; i < NX; i++) for (int l = 0; l < NZ; l++) { double a = 0.0; for (int j = 0; j < NX; j++) a += Pn[i][j] * AB[j][l]; W[i][l] = a; }
            for (int a = 0; a < NZ; a++) {
                for (int b = 0; b < NZ; b++) {
                    double s = c[C_H + (a <= b ? J2::hi(a, b) : J2::hi(b, a))];
                    for (int i = 0; i < NX; i++) s += AB[i][a] * W[i][b];
                    Mm[a][b] = s;
                }
                Mm[a][a] += row(R_DGV, k)[a];
                double s = row(R_HV, k)[a];
                for (int i = 0; i < NX; i++) s += AB[i][a] * pr[i];
                mv[a] = s;
            }
            // eliminate the controls: Cholesky of M_uu (pivot <= 0: wrong inertia), K = M_uu^-1 M_ux, kf = M_uu^-1 m_u
            double L[NU][NU], Kk[NU][NX], kf[NU];
            for (int a = 0; a < NU; a++)
                for (int b = 0; b <= a; b++) {
                    double sacc = Mm[NX + a][NX + b];
                    for (int t = 0; t < b; t++) sacc -= L[a][t] * L[b][t];
                    if (a == b) {
                        if (!(sacc > 0.0) || !(sacc < NMPC_INF)) return false;
                        L[a][a] = sqrt(sacc);
                    } else L[a][b] = sacc / L[b][b];
                }
            for (int j = 0; j <= NX; j++) {   // columns of M_ux, then m_u
                double y[NU];
                for (int a = 0; a < NU; a++) {
                    double sacc = j < NX ? Mm[NX + a][j] : mv[NX + a];
                    for (int t = 0; t < a; t++) sacc -= L[a][t] * y[t];
                    y[a] = sacc / L[a][a];
                }
                for (int a = NU - 1; a >= 0; a--) {
                    double sacc = y[a];
                    for (int t = a + 1; t < NU; t++) sacc -= L[t][a] * y[t];
                    y[a] = sacc / L[a][a];
                }
                for (int a = 0; a < NU; a++) { if (j < NX) Kk[a][j] = y[a]; else kf[a] = y[a]; }
            }
            for (int i = 0; i < NX; i++) {   // P = M_xx - M_xu K,  p = m_x - M_xu kf
                for (int j = 0; j < NX; j++) { double sacc = Mm[i][j]; for (int a = 0; a < NU; a++) sacc -= Mm[i][NX + a] * Kk[a][j]; Mm[i][j] = sacc; }
                double sacc = mv[i];
                for (int a = 0; a < NU; a++) sacc -= Mm[i][NX + a] * kf[a];
                mv[i] = sacc;
            }
            double *cw = cst(k);
            for (int i = 0; i < NX; i++) {
                for (int j = 0; j < NX; j++) { Pn[i][j] = 0.5 * (Mm[i][j] + Mm[j][i]); cw[C_P + i * NX + j] = Pn[i][j]; }
                pn[i] = mv[i]; row(R_LIN, k)[i] = pn[i];
            }
            for (int u = 0; u < NU; u++) { for (int j = 0; j < NX; j++) cw[C_K + u * NX + j] = Kk[u][j]; cw[C_KF + u] = kf[u]; }
        }
        return true;
    }

    __device__ __noinline__ void forward(double mu, double tau, int rdz, int rds, int rytc, int rytd, StepInfo &si)
    {
        double ap = 0.0, az = 0.0, gbd = 0.0, tiny = 0.0, dx[NX], du[NU];
        for (int i = 0; i < NX; i++) dx[i] = INIT_ROWS ? row(R_RC, 0)[i] : 0.0;   // dx_0 = x0bar - X_0 (or 0: X_0 is a parameter)
        for (int k = 0; k <= N; k++) {
            const double *c = cst(k);
            for (int i = 0; i < NX; i++) {   // multiplier of the rows that define X_k: the co-state P_k dx + p_k
                double a = row(R_LIN, k)[i];
                for (int j = 0; j < NX; j++) a += c[C_P + i * NX + j] * dx[j];
                row(rytc, k)[i] = a;
            }
            for (int u = 0; u < NU; u++) {
                double a = 0.0;
                if (k < N) { a = c[C_KF + u]; for (int j = 0; j < NX; j++) a += c[C_K + u * NX + j] * dx[j]; }
                du[u] = -a;
            }
            for (int l = 0; l < LD; l++) {
                const double dzl = l < NX ? dx[l] : (l < NZ ? du[l - NX] : 0.0);
                row(rdz, k)[l] = dzl;
                if (valid(k, l)) {
                    const double z = row(R_Z, k)[l];
                    WS::slack_step_terms(z, dzl, row(R_BL, k)[l], row(R_BU, k)[l], row(R_ZL, k)[l], row(R_ZU, k)[l], mu, ap, az);
                    gbd += row(R_GX, k)[l] * dzl; tiny = fmax(tiny, fabs(dzl) / (1.0 + fabs(z)));
                }
            }
            if (k < N) {
                for (int i = 0; i < LD; i++) {   // slack steps and inequality multipliers of the rows on X_k
                    double ds = 0.0, ytd = 0.0;
                    if (i < ni && qact(k, i)) {
                        const double *ci = cin(k, i);
                        const double gs = row(R_GS, k)[i], s = row(R_S, k)[i];
                        ds = row(R_RD, k)[i];
                        for (int a = 0; a < NX; a++) ds += ci[1 + a] * dx[a];
                        ytd = row(R_DQ, k)[i] * ds + gs;
                        WS::slack_step_terms(s, ds, row(R_DL, k)[i], row(R_DU, k)[i], row(R_VL, k)[i], row(R_VU, k)[i], mu, ap, az);
                        gbd += gs * ds; tiny = fmax(tiny, fabs(ds) / (1.0 + fabs(s)));
                    }
                    row(rds, k)[i] = ds; row(rytd, k)[i] = ytd;
                }
                double dn[NX];
                for (int i = 0; i < NX; i++) {
                    double a = row(R_RC, k + 1)[i];
                    for (int j = 0; j < NX; j++) a += c[C_J + i * NZ + j] * dx[j];
                    for (int u = 0; u < NU; u++) a += c[C_J + i * NZ + NX + u] * du[u];
                    dn[i] = a;
                }
                for (int i = 0; i < NX; i++) dx[i] = dn[i];
            }
        }
        si.ap = ap > tau ? tau / ap : 1.0; si.az = az > tau ? tau / az : 1.0; si.gbd = gbd; si.tiny = tiny;
    }

    __device__ __forceinline__ double mult_upd(double m, double az, double mu, double sl_old, double sl_new, double dv_signed) const
    {
        const double ks = P.o.kappa_sigma, r = 1.0 / sl_old, cc = mu / sl_new;
        return fmax(fmin(m + az * (mu * r - m + m * r * dv_signed), ks * cc), cc / ks);
    }
    __device__ __noinline__ void accept(double alpha, double az, double mu, int rdz, int rds, int rytc, int rytd)
    {
        for (int k = 0; k <= N; k++)
            for (int l = 0; l < LD; l++) {
                if (valid(k, l)) {
                    const double z = row(R_Z, k)[l], dz = row(rdz, k)[l], lo = row(R_BL, k)[l], hi = row(R_BU, k)[l], zn = z + alpha * dz;
                    if (lo > -NMPC_INF) row(R_ZL, k)[l] = mult_upd(row(R_ZL, k)[l], az, mu, z - lo, zn - lo, -dz);
                    if (hi < NMPC_INF) row(R_ZU, k)[l] = mult_upd(row(R_ZU, k)[l], az, mu, hi - z, hi - zn, dz);
                    row(R_Z, k)[l] = zn;
                }
                if (l < NX && k >= kfirst()) { const double yc = row(R_YC, k)[l]; row(R_YC, k)[l] = yc + alpha * (row(rytc, k)[l] - yc); }
                if (l < ni && k < N && qact(k, l)) {
                    const double s = row(R_S, k)[l], ds = row(rds, k)[l], lo = row(R_DL, k)[l], hi = row(R_DU, k)[l], sn = s + alpha * ds;
                    if (lo > -NMPC_INF) row(R_VL, k)[l] = mult_upd(row(R_VL, k)[l], az, mu, s - lo, sn - lo, -ds);
                    if (hi < NMPC_INF) row(R_VU, k)[l] = mult_upd(row(R_VU, k)[l], az, mu, hi - s, hi - sn, ds);
                    row(R_S, k)[l] = sn;
                    const double yd = row(R_YD, k)[l];
                    row(R_YD, k)[l] = yd + alpha * (row(rytd, k)[l] - yd);
                }
            }
    }
    __device__ __noinline__ void accept_primal(double alpha, int rdz, int rds)
    {
        for (int k = 0; k <= N; k++)
            for (int l = 0; l < LD; l++) {
                if (valid(k, l)) row(R_Z, k)[l] += alpha * row(rdz, k)[l];
                if (l < ni && k < N && qact(k, l)) row(R_S, k)[l] += alpha * row(rds, k)[l];
            }
    }
    __device__ __noinline__ void resto_reset(double mu)
    {
        const double ks = P.o.kappa_sigma;
        auto clip = [=](double m, double s2) { return fmax(fmin(m, ks * mu / s2), mu / (ks * s2)); };
        for (int k = 0; k <= N; k++)
            for (int l = 0; l < LD; l++) {
                if (valid(k, l)) {
                    const double z = row(R_Z, k)[l], lo = row(R_BL, k)[l], hi = row(R_BU, k)[l];
                    if (lo > -NMPC_INF) row(R_ZL, k)[l] = clip(row(R_ZL, k)[l], z - lo);
                    if (hi < NMPC_INF) row(R_ZU, k)[l] = clip(row(R_ZU, k)[l], hi - z);
                }
                row(R_YC, k)[l] = 0.0; row(R_YD, k)[l] = 0.0;
                if (l < ni && k < N && qact(k, l)) {
                    const double s = row(R_S, k)[l], lo = row(R_DL, k)[l], hi = row(R_DU, k)[l];
                    if (lo > -NMPC_INF) row(R_VL, k)[l] = clip(row(R_VL, k)[l], s - lo);
                    if (hi < NMPC_INF) row(R_VU, k)[l] = clip(row(R_VU, k)[l], hi - s);
                }
            }
    }
    // restoration candidate: integrate the current controls forward from the initial state (every equality row becomes zero)
    __device__ __noinline__ void rollout_project()
    {
        const nmpc_opts &o = P.o;
        double zt[LD];
        for (int l = 0; l < LD; l++) zt[l] = row(R_Z, 0)[l];
        if (INIT_ROWS)
            for (int i = 0; i < NX; i++) zt[i] = WS::push_in(Model::x0bar(ctx, i) + row(R_CE, 0)[i], row(R_BL, 0)[i], row(R_BU, 0)[i], o.bound_push, o.bound_frac);
        for (int k = 0; k <= N; k++) {
            for (int l = 0; l < LD; l++) row(R_DZ, k)[l] = valid(k, l) ? zt[l] - row(R_Z, k)[l] : 0.0;
            if (k < N) {
                model(k, zt);
                for (int i = 0; i < LD; i++)
                    row(R_DS, k)[i] = (i < ni && qact(k, i)) ? WS::push_in(cin(k, i)[0], row(R_DL, k)[i], row(R_DU, k)[i], o.bound_push, o.bound_frac) - row(R_S, k)[i] : 0.0;
                for (int i = 0; i < NX; i++) zt[i] = WS::push_in(cst(k)[C_F + i] - Model::EQ_SIGN * row(R_CE, k + 1)[i], row(R_BL, k + 1)[i], row(R_BU, k + 1)[i], o.bound_push, o.bound_frac);
                for (int u = 0; u < NU; u++) zt[NX + u] = k + 1 < N ? row(R_Z, k + 1)[NX + u] : 0.0;
            }
        }
    }
    __device__ __noinline__ void soc_begin()
    {
        for (int k = 0; k <= N; k++)
            for (int l = 0; l < LD; l++) { row(R_CSOC, k)[l] = l < NX ? row(R_RC, k)[l] : 0.0; row(R_DSOC, k)[l] = (l < ni && k < N) ? row(R_RD, k)[l] : 0.0; }
    }
    __device__ double mult_absmax()
    {
        double m = 0.0;
        for (int k = 0; k <= N; k++) {
            if (k >= kfirst()) for (int i = 0; i < NX; i++) m = fmax(m, fabs(row(R_YC, k)[i]));
            if (k < N) for (int i = 0; i < ni; i++) m = fmax(m, fabs(row(R_YD, k)[i]));
        }
        return m;
    }
    __device__ void mult_zero() { for (int k = 0; k <= N; k++) for (int l = 0; l < LD; l++) { row(R_YC, k)[l] = 0.0; row(R_YD, k)[l] = 0.0; } }

    __device__ bool filter_ok(double th, double ph) const
    {
        for (int i = 0; i < fn; i++)
            if (!(th < fth[i] || ph < fph[i])) return false;
        return true;
    }
    __device__ __noinline__ void filter_add(double th, double ph)
    {
        int m = 0;
        for (int i = 0; i < fn; i++)
            if (!(fth[i] >= th && fph[i] >= ph)) { fth[m] = fth[i]; fph[m] = fph[i]; m++; }
        if (m == NMPC_FILTER_CAP_SMALL) { for (int i = 1; i < m; i++) { fth[i - 1] = fth[i]; fph[i - 1] = fph[i]; } m--; n_evict++; }
        fth[m] = th; fph[m] = ph; fn = m + 1;
    }
    __device__ bool trial_ok(double th_t, double ph_t, double theta, double phi, double theta_max, double theta_min, double gbd,
                             double alpha_test, bool ftype) const
    {
        if (!(WS::fin(th_t) && WS::fin(ph_t)) || !WS::cmp_le(th_t, theta_max, theta)) return false;
        bool ok;
        if (ftype && theta <= theta_min) ok = WS::cmp_le(ph_t - phi, 1e-8 * alpha_test * gbd, phi);
        else ok = WS::cmp_le(th_t, (1.0 - 1e-5) * theta, theta) || WS::cmp_le(ph_t - phi, -1e-8 * theta, phi);
        return ok && filter_ok(th_t, ph_t);
    }

    // outputs in the reference layout and sign conventions (g = F - X_next, and X_0 - x0bar for the initial rows)
    __device__ __noinline__ void write_outputs(int st, int iter, double E0, double pinf, double dinf, double c0, double mu)
    {
        const long long n = Model::n(N, ctx.nobs), mg = Model::mg(N, ctx.nobs);
        double *x = P.x + inst * n;
        double fo = 0.0;
        for (int k = 0; k <= N; k++)
            for (int l = 0; l < (k < N ? NZ : NX); l++) {
                x[Model::xidx(ctx, k, l)] = row(R_Z, k)[l];
                if (P.lam_x) P.lam_x[inst * n + Model::xidx(ctx, k, l)] = valid(k, l) ? (row(R_ZU, k)[l] - row(R_ZL, k)[l]) / df : 0.0;
            }
        for (int k = 0; k < N; k++) { model(k, row(R_Z, k)); fo += cst(k)[C_Q]; }
        // A fixed initial state is a parameter (IPOPT's make_parameter): its bound multiplier is -(grad f + J' lam_g), the
        // cost's sensitivity to X_0, so that grad f + J' lam_g + lam_x = 0 holds in every component.
        if (P.lam_x && fixed0)
            for (int l = 0; l < NX; l++) {
                double r = df * cst(0)[C_GQ + l];
                for (int i = 0; i < NX; i++) r += cst(0)[C_J + i * NZ + l] * row(R_YC, 1)[i];
                for (int i = 0; i < ni; i++) r += cin(0, i)[1 + l] * row(R_YD, 0)[i];
                P.lam_x[inst * n + Model::xidx(ctx, 0, l)] = -r / df;
            }
        for (int k = kfirst(); k <= N; k++)
            for (int i = 0; i < NX; i++) {
                const long long r = inst * mg + Model::grow_eq(ctx, k, i);
                const double sgn = k == 0 ? -1.0 : (double)Model::EQ_SIGN;   // the initial rows are reported as X_0 - x0bar
                if (P.g) P.g[r] = sgn * ((k == 0 ? Model::x0bar(ctx, i) : cst(k - 1)[C_F + i]) - row(R_Z, k)[i]);
                if (P.lam_g) P.lam_g[r] = sgn * row(R_YC, k)[i] / df;
            }
        for (int k = 0; k < N; k++)
            for (int i = 0; i < ni; i++) {
                const long long r = inst * mg + Model::grow_in(ctx, k, i);
                if (P.g) P.g[r] = cin(k, i)[0];
                if (P.lam_g) P.lam_g[r] = row(R_YD, k)[i] / df;
            }
        if (P.f) P.f[inst] = fo;
        if (P.status) P.status[inst] = st;
        if (P.iters) P.iters[inst] = iter;
        if (P.stats) {
            double *sp = P.stats + (long long)inst * NMPC_NSTATS;
            sp[NMPC_ST_KKT_ERR] = E0; sp[NMPC_ST_PRIMAL_INF] = pinf; sp[NMPC_ST_DUAL_INF] = dinf; sp[NMPC_ST_COMPL] = c0;
            sp[NMPC_ST_MU] = mu; sp[NMPC_ST_N_REG] = n_reg; sp[NMPC_ST_N_RESTO] = n_resto; sp[NMPC_ST_N_SOC] = n_soc;
            sp[NMPC_ST_N_FACTOR] = n_fact; sp[NMPC_ST_N_LS] = n_ls; sp[NMPC_ST_FILTER_EVICT] = n_evict;
        }
    }
    __device__ void run() { ipm_run(*this); }
};

// one thread per instance
template <class Model>
__global__ void __launch_bounds__(64) solve_kernel_small_ocp(const NmpcSolveParams P)
{
    for (int inst = blockIdx.x * blockDim.x + threadIdx.x; inst < P.B; inst += gridDim.x * blockDim.x) {
        ThreadSolver<Model> s(P, P.ws + (long long)inst * P.ws_stride);
        s.setup(inst);
        s.run();
    }
}
