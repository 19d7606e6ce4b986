// Warp-per-instance primal-dual interior-point solver for the Nr-robot unicycle NMPC NLP.
//
// Replaces, for one instance, everything behind the reference's
//     sol = solver(x0=, p=, lbx=, ubx=, lbg=, ubg=)     centralized_six_robots_implementation.py:432
// i.e. CasADi's derivative evaluation (K1), IPOPT's filter line-search interior-point iteration
// (K2) and the MUMPS factorisation of the KKT system (K3, done here as a stage-wise Riccati
// sweep).  NLP definition: same file :207-352 (cost :314, defects/distances :282-331, bounds
// :349-352); algorithm: Waechter & Biegler 2006 with IPOPT's default options (SURVEY.md App. B).
//
// Mapping: lane l of the warp owns variable l of the stage vector z_k = [X_k ; U_k]
// (5 Nr <= 30 lanes), pair row q of an inequality block (lanes < M), and COLUMN l of the
// (5Nr+1) x 5Nr bordered stage KKT matrix, which lives in registers.  Eliminating the control
// block is a symmetric sweep: the pivot row is exchanged through shared memory, the rank-1
// update is 5Nr+1 independent DFMAs per lane.  Iterates, steps and the Riccati factors stream
// through a per-warp scratch area in global memory in [stage][32-lane] rows (256 B, coalesced).
//
// The file is written against the small `wp::` interface (warp_prims.cuh) so that the tests can
// step the same source through a CPU fibre emulation of a warp (tests/emul/).
#pragma once
#include <type_traits>
#include "nmpc_internal.h"
#include "ipm_driver.cuh"

#ifndef NMPC_INF
#define NMPC_INF ((double)INFINITY)
#endif


// Inside a noinline pass the solver object lives in local memory; shadow the members that the pass
// uses with locals so they are loaded once, and re-derive the pointers with their address spaces
// (shared / global) so the compiler emits LDS/LDG instead of generic loads.
#define NMPC_LOCALS                                                                                   \
    double *const sm = wp::shared_ptr(this->sm);                                                      \
    double *const ws = wp::global_ptr(this->ws);                                                      \
    const double *const br = wp::global_ptr(this->br);                                                 \
    const int N = this->N, S = this->S, l = this->l, rob = this->rob, comp = this->comp,               \
              pi = this->pi, pj = this->pj;                                                            \
    const bool isx = this->isx, isu = this->isu, isz = this->isz, isq = this->isq;                     \
    const double T = this->T, df = this->df, xs_l = this->xs_l, qw = this->qw, x0bar_l = this->x0bar_l; \
    const int nobs = OBS ? this->nobs : 0, family = OBS ? this->family : 0;                              \
    const bool isobs = OBS && this->isobs;                                                              \
    const double *const qob = OBS ? wp::global_ptr(this->qob) : nullptr;                                \
    const long long qos = OBS ? this->qos : 0;                                                          \
    (void)nobs; (void)family; (void)isobs; (void)qob; (void)qos;                                         \
    (void)sm; (void)ws; (void)br; (void)N; (void)S; (void)l;                                            \
    (void)rob; (void)comp; (void)pi; (void)pj; (void)isx; (void)isu; (void)isz; (void)isq; (void)T;    \
    (void)df; (void)xs_l; (void)qw; (void)x0bar_l;                                                     \
    auto row = [=](int r, int k) -> double * { return ws + ((long long)k * R_COUNT + r) * LW; };       \
    auto frow = [=](int k, int i) -> double * { return ws + ((long long)k * R_COUNT + R_F0 + i) * LW; }; \
    auto brow = [=](int x, int k) -> const double * { return br + ((long long)k * NMPC_BR_COUNT + x) * LW; }; \
    (void)brow;                                                                                        \
    auto zvalid = [=](int k) -> bool { return l < (k < N ? NZ : NS); };                                \
    auto gradf = [=](int k, double z, double xr) -> double { return (k < N && isz) ? qw * (z - xr) : 0.0; }; \
    (void)row; (void)frow; (void)zvalid; (void)gradf;

struct alignas(16) NmpcD2 { double x, y; };   // one 128-bit shared-memory load
#ifndef NMPC_PIVOT_UNROLL
#define NMPC_PIVOT_UNROLL 1   // 2: both pivot-row buffers get compile-time addresses (6 % fewer instructions per pivot) but the loop body
                              // doubles; measured slower (43.8 k against 46.5 k solves/s): instruction fetch, not issue, is the limit
#endif
#ifndef NMPC_XBATCH
#define NMPC_XBATCH 3   // pairs of pivot-row entries per batch of the sweep's state-row update (see factor())
#endif

// OBS: the static-obstacle family (obstacle rows after the pair rows).  A separate instantiation: the generalised row geometry and
// the wider addend tables cost the pair-only benchmark path 8 % when they are merely switched off at run time (measured).
// TRK: trajectory tracking (nmpc_create_tracking), the centralized family with a per-stage reference Z[k] = [xr_k; ur_k] in p
// (p = [x0bar; Z[0..N-1]]) instead of one setpoint xs.  The reference is copied once per solve into row R_REF of each stage record
// (lane l: Z[k][l], lanes >= NZ and record N: 0), where the passes load it with the rows they already stage; the instantiations
// without TRK keep the setpoint in a register (xs_l) and have no R_REF row.
template <int NR, bool OBS = false, bool TRK = false>
struct WarpSolver {
    static constexpr int NS = 3 * NR, NC = 2 * NR, NZ = 5 * NR, M = NR * (NR - 1) / 2;
    static constexpr int LIN = NZ, NM = NZ + 1;
    // lanes per instance ("team"): one warp up to 6 robots; two warps (one 64-thread CTA) for 7..11 robots
    static constexpr int LW = (NZ + 1 <= 32) ? 32 : 64;
    static constexpr int CFS = LW / 4;        // stride of the four coefficient groups inside a R_COEF row
    static constexpr int LPR = LW / 16;       // 128-byte lines per scratch row
    static constexpr int NRP = (NR <= 8) ? 8 : 16, MP = (M <= 16) ? 16 : 64;
    // static circular obstacles (family F of the reference, first_scenario_mpc_obstacle_avoidance.py:96-152): nobs rows per robot and
    // stage after the M pair rows, one lane each, so Nr * nobs <= LW - M on this path
    static constexpr int NOBS_MAX = OBS ? (LW - M) / NR : 0, TCOLS = NR + NOBS_MAX;
    static_assert(NZ + 1 <= 64 && M <= LW, "at most 10 robots on the lane-per-column path");
    // Scratch layout: one RECORD of R_COUNT rows (LW doubles each) per stage, records consecutive in memory.  The rows are ordered
    // so that what a pass stages for one stage is two contiguous ranges: rows indexed by the stage k (from record k) and rows indexed
    // by the block k + 1 (from record k + 1):
    //     factorisation:  record k  [R_REF .. R_ZU]                  record k + 1  [R_YC .. R_VU]
    //     forward pass:   record k  [R_Z .. R_F0 + NS - 1]           record k + 1  [R_S .. R_DQ]
    // (round 1 kept one array per row, [row][stage][LW]: the 16 rows a stage needs were 16 separate 256-byte pieces 5 KB apart).
    // The (relaxed) bound rows are laid out the same way by prep_bounds_kernel ([stage][BL, BU, CE, DL, DU][LW]); they are shared by the
    // batch unless bounds_batched and stay L2 resident (copying them into every instance's records cost 10 MB of DRAM traffic per solve).
    enum Row {
        R_REF, R_TRIG2 = R_REF + (TRK ? 1 : 0),
        R_TRIG, R_Z, R_ZL, R_ZU, R_LIN, R_DG, R_GX, R_COEF, R_F0,                  // R_F0 .. R_F0 + NS - 1: Riccati factor rows
        R_YC = R_F0 + NS, R_YD, R_CSOC, R_DSOC, R_S, R_VL, R_VU, R_RC, R_GS, R_GXQ, R_GYQ, R_RD, R_DQ,
        R_DZ, R_DZ2, R_YTC, R_YTC2, R_DS, R_DS2, R_YTD, R_YTD2,
        R_COUNT
    };
    // slots of the factorisation's staging buffer (sm + SM_STG): rows [R_REF .. R_ZU] of record k, bound rows [BL, BU] of stage k,
    // rows [R_YC .. R_VU] of record k + 1, bound rows [CE, DL, DU] of block k + 1  (R_REF / FS_REF: TRK only, else an alias of
    // R_TRIG2 / FS_TRIG2)
    enum { FS_REF, FS_TRIG2 = FS_REF + (TRK ? 1 : 0),
           FS_TRIG, FS_Z, FS_ZL, FS_ZU, FS_BL, FS_BU, FS_YC, FS_YD, FS_CSOC, FS_DSOC, FS_S, FS_VL, FS_VU, FS_CE, FS_DL, FS_DU, FS_COUNT };
    // slots of the forward pass's staging buffer (the whole big region): rows [R_Z .. last factor row] of record k, [BL, BU] of stage k,
    // rows [R_S .. R_DQ] of record k + 1, [DL, DU] of block k + 1
    enum { WS_Z, WS_ZL, WS_ZU, WS_LIN, WS_DG, WS_GX, WS_COEF, WS_F0, WS_BL = WS_F0 + NS, WS_BU,
           WS_S, WS_VL, WS_VU, WS_RC, WS_GS, WS_GXQ, WS_GYQ, WS_RD, WS_DQ, WS_DL, WS_DU, WS_COUNT };
    static_assert(R_ZU - R_REF == FS_ZU - FS_REF && R_TRIG2 - R_REF == FS_TRIG2 - FS_REF && R_VU - R_YC == FS_VU - FS_YC &&
                  R_F0 + NS - 1 - R_Z == WS_F0 + NS - 1 - WS_Z &&
                  R_DQ - R_S == WS_DQ - WS_S && NMPC_BR_BU == NMPC_BR_BL + 1 && NMPC_BR_DL == NMPC_BR_CE + 1 && NMPC_BR_DU == NMPC_BR_DL + 1,
                  "staging slots follow the record layouts");
    // shared-memory carve-up (doubles, per team): small buffers that live for the whole solve, then one big region that the
    // factorisation and the forward pass carve up differently (they never run at the same time)
    enum {
        PLD = NS + 3,  // leading dimension of the P broadcast buffer: 3Nr columns of P, the pr column, 2 zero columns
        TSZ = NR * TCOLS, // one addend table of the stage-matrix build (rows: robots; columns: robots, then this robot's obstacles), see factor()
        SM_ZB = 0, SM_DZB = SM_ZB + LW, SM_RCB = SM_DZB + LW, SM_PRB = SM_RCB + LW, SM_HB = SM_PRB + LW,
        SM_CS = SM_HB + LW, SM_SN = SM_CS + NRP, SM_C4 = SM_SN + NRP,   // c4[4 i ..]: a_i, b_i, T cos, T sin of robot i (one 32-byte record)
        SM_CRS = SM_C4 + 4 * NRP, SM_THD = SM_CRS + NRP,
        SM_MISC = SM_THD + NRP,
        SM_MBAR = SM_MISC + 4,           // the team's mbarrier (8 bytes) for the bulk-copy staging
        SM_RED = SM_MISC + 8,            // cross-warp reduction scratch (two-warp teams)
        SM_BIG = SM_RED + 8,
        // -- factorisation view of the big region
        SM_COL = SM_BIG,                 // two pivot-row buffers, each LW values + LW reciprocals
        SM_PB = SM_COL + 4 * LW,
        SM_TT = SM_PB + ((NS * PLD + 1) & ~1),     // 8 addend tables [NR][NR], the gradient rows HH[5][NR], a row of zeros
        TT_DOUBLES = (8 * TSZ + 6 * NR + 1) & ~1,
        STG_ROWS = FS_COUNT,
        SM_STG = SM_TT + TT_DOUBLES,     // rows of the NEXT stage, copied asynchronously (cp.async) while this one is processed
        BIG_FACTOR = SM_STG + STG_ROWS * LW - SM_BIG,
        // -- forward view: WS_COUNT staging rows from SM_BIG
        BIG_FORWARD = WS_COUNT * LW,
        SM_DOUBLES = SM_BIG + (BIG_FACTOR > BIG_FORWARD ? BIG_FACTOR : BIG_FORWARD)
    };
    static_assert((int)WS_COUNT <= 64 && (SM_BIG & 1) == 0 && (SM_STG & 1) == 0 && (SM_DOUBLES & 1) == 0 && (SM_C4 & 3) == 0, "shared-memory layout");

    // Staging of a pass: up to four contiguous ranges of rows per stage, each ONE TMA bulk copy (cp.async.bulk global -> shared) issued
    // by lane 0 of the team, all of them completing on the team's mbarrier (sm[SM_MBAR]); stage_wait() is the consumer side.  (The
    // first record-layout version copied the ranges with cp.async, 16 bytes per lane: 10 + 20 loop iterations per stage pair.)
    static NMPC_DEV void bulk_rows(double *bar, double *dst, const double *src, int nrows)
    {
        wp::bulk_g2s(dst, src, (unsigned)(nrows * LW * sizeof(double)), bar);
    }
    // once per team and kernel: the staging barrier (one arriving thread per phase: the issuing lane's expect_tx)
    NMPC_DEV void init_team()
    {
        if (wp::team_lane(LW) == 0) wp::mbar_init(wp::shared_ptr(this->sm) + SM_MBAR);
        mbar_phase = 0;
        tsync();
    }
    NMPC_DEV void stage_wait()
    {
        wp::mbar_wait(wp::shared_ptr(this->sm) + SM_MBAR, (unsigned)mbar_phase);
        mbar_phase ^= 1;
    }
    // per-slot scratch: the stage records, then the filter (NMPC_FILTER_CAP theta values, then as many phi values)
    static NMPC_HD long long ws_doubles(int N) { return (long long)R_COUNT * (N + 1) * LW + 2 * NMPC_FILTER_CAP; }

    const NmpcSolveParams &P;
    double *sm, *ws;
    const double *br;   // this instance's bound rows, [stage][BL, BU, CE, DL, DU][LW]
    int N, S, l, rob, comp, pi, pj, inst, fn;
    // cos/sin rows of the iterate (r_trig is R_TRIG or R_TRIG2; the other one receives the trial points).  When a step is
    // accepted at the trial point evaluated last, its rows BECOME the iterate's (swap) and no sincos is recomputed.
    int r_trig, t2_rdz;
    int mbar_phase;   // parity of the staging mbarrier's current phase
    bool trig_valid;
    double t2_alpha;
    bool isx, isu, isz, isq;
    // inequality rows of a block: lanes < M are the pair rows (pi, pj); lanes M .. M + Nr nobs - 1 the obstacle rows, robot-major
    // (row M + i nobs + o: robot pi = i against obstacle o); family 1 = the obstacle scripts' g layout.  The obstacle table of stage k
    // ([nobs][3] = centre x, y, clearance) is qtab + k qos: the handle's static table (qos = 0) or the instance's block of p;
    // qob = qtab + 3 o: this lane's obstacle at stage 0
    int nobs, family;
    bool isobs;
    const double *qtab, *qob;
    long long qos;
    double T, df, xs_l, qw, x0bar_l, ny_nzb, nzb_cnt;
    int n_reg, n_resto, n_soc, n_fact, n_ls;

    NMPC_DEV WarpSolver(const NmpcSolveParams &p, double *smem, double *wsp) : P(p), sm(smem), ws(wsp) {}

    // team-wide barrier and all-reduce (a team is one warp, or the two warps of a 64-thread CTA)
    static NMPC_DEV void tsync() { if (LW == 32) wp::sync(); else wp::sync_team64(); }
    NMPC_DEV double tred(double v, int op) const
    {
        double r = op == 0 ? wp::red_sum(v) : (op == 1 ? wp::red_max(v) : wp::red_min(v));
        if (LW == 64) {
            double *sc = wp::shared_ptr(this->sm) + SM_RED;
            const int tl = wp::team_lane(LW);
            tsync();
            if ((tl & 31) == 0) sc[tl >> 5] = r;
            tsync();
            const double a = sc[0], b = sc[1];
            r = op == 0 ? a + b : (op == 1 ? fmax(a, b) : fmin(a, b));
        }
        return r;
    }
    NMPC_DEV double tred_sum(double v) const { return tred(v, 0); }
    NMPC_DEV double tred_max(double v) const { return tred(v, 1); }
    NMPC_DEV double tred_min(double v) const { return tred(v, 2); }

    NMPC_DEV double *row(int r, int k) const { return ws + ((long long)k * R_COUNT + r) * LW; }
    NMPC_DEV double *frow(int k, int i) const { return ws + ((long long)k * R_COUNT + R_F0 + i) * LW; }
    NMPC_DEV bool zvalid(int k) const { return l < (k < N ? NZ : NS); }
    static NMPC_DEV int pairidx(int a, int b) { return a * (2 * NR - a - 1) / 2 + (b - a - 1); }
    static NMPC_DEV bool fin(double v) { return v > -NMPC_INF && v < NMPC_INF; }
    // One inequality row evaluated on a stage vector zr: value, gradient w.r.t. (x_pi, y_pi) (negated for robot pj of a pair row)
    // and its own second derivatives.  Pair rows: squared distance (centralized_six_robots_implementation.py:288-306); obstacle
    // rows: sqrt((x - ox)^2 + (y - oy)^2) - clearance (first_scenario_mpc_obstacle_avoidance.py:96-99,125), ob = (ox, oy, clearance)
    // of the row's obstacle at the stage of zr.
    struct RowG { double dv, gx, gy, hxx, hyy, hxy; };
    static NMPC_DEV RowG rowg(const double *zr, int pi, int pj, bool isobs, const double *ob)
    {
        RowG r;
        if (isobs) {
            const double dx = zr[3 * pi] - ob[0], dy = zr[3 * pi + 1] - ob[1];
            const double rho = sqrt(dx * dx + dy * dy), ir = 1.0 / rho;
            r.gx = dx * ir; r.gy = dy * ir; r.dv = rho - ob[2];
            r.hxx = (1.0 - r.gx * r.gx) * ir; r.hyy = (1.0 - r.gy * r.gy) * ir; r.hxy = -r.gx * r.gy * ir;
        } else {
            const double dx = zr[3 * pi] - zr[3 * pj], dy = zr[3 * pi + 1] - zr[3 * pj + 1];
            r.dv = dx * dx + dy * dy; r.gx = 2.0 * dx; r.gy = 2.0 * dy; r.hxx = 2.0; r.hyy = 2.0; r.hxy = 0.0;
        }
        return r;
    }

    // ---------------------------------------------------------------------------------------
    NMPC_DEV void setup(int instance)
    {
        inst = instance; N = P.N; S = N + 1; T = P.T; l = wp::team_lane(LW);
        nobs = OBS ? P.nobs : 0; family = OBS ? P.family : 0;
        isx = l < NS; isu = l >= NS && l < NZ; isz = l < NZ; isq = l < M + NR * nobs; isobs = isq && l >= M;
        qos = 0; qtab = qob = nullptr;
        rob = isx ? l / 3 : (isu ? (l - NS) / 2 : 0);
        comp = isx ? l % 3 : (isu ? (l - NS) % 2 : 0);
        pi = 0; pj = 0;
        if (isobs) {
            pi = (l - M) / nobs; pj = pi;   // pj = pi: the "other robot" terms of a pair row cancel for an obstacle row
        } else if (isq) {
            int q = 0;
            for (int a = 0; a < NR; a++)
                for (int b = a + 1; b < NR; b++) { if (q == l) { pi = a; pj = b; } q++; }
        }
        br = P.brows + (long long)inst * P.bstride;
        const double *pp = P.p + (long long)inst * ((OBS || TRK) ? P.np : 2 * NS);
        if (OBS) {   // obstacles in p: [N][nobs][3] after x0bar and xs (TRK: after x0bar and Z[0..N-1]), one table per stage;
                     // else the handle's table at every stage
            qtab = P.obs_in_p ? pp + (TRK ? NS + N * NZ : 2 * NS) : P.obs; qos = P.obs_in_p ? 3 * nobs : 0;
            if (isobs) qob = qtab + 3 * ((l - M) % nobs);
        }
        x0bar_l = isx ? pp[l] : 0.0;
        xs_l = (isx && !TRK) ? pp[NS + l] : 0.0;   // TRK: the reference is in the R_REF rows (init_point)
        qw = isx ? 2.0 * P.Q[comp] : (isu ? 2.0 * P.R[comp] : 0.0);
        df = 1.0; fn = 0;
        n_reg = n_resto = n_soc = n_fact = n_ls = 0;
        if (l == 0) sm[SM_MISC + 2] = 0.0;   // filter evictions (NMPC_ST_FILTER_EVICT)
        tsync();
    }

    // gradient of the stage cost of variable l at stage k; xr: its reference (xs_l, or row R_REF of record k with TRK)
    NMPC_DEV double gradf(int k, double z, double xr) const { return (k < N && isz) ? qw * (z - xr) : 0.0; }

    static NMPC_DEV double push_in(double x, double lo, double hi, double k1, double k2)
    {
        bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
        if (hl && hu) {
            double pl = fmin(k1 * fmax(1.0, fabs(lo)), k2 * (hi - lo));
            double pu = fmin(k1 * fmax(1.0, fabs(hi)), k2 * (hi - lo));
            x = fmax(x, lo + pl); x = fmin(x, hi - pu);
        } else if (hl) x = fmax(x, lo + k1 * fmax(1.0, fabs(lo)));
        else if (hu) x = fmin(x, hi - k1 * fmax(1.0, fabs(hi)));
        return x;
    }

    // starting point: objective scaling, push into bounds, slacks, bound multipliers
    NMPC_PASS void init_point()
    {
        NMPC_LOCALS
        const double *x0 = P.x0 + (long long)inst * (NS * S + NC * N);
        const nmpc_opts &o = P.o;
        double gmax = 0.0;
        const double *zref = TRK ? P.p + (long long)inst * P.np + NS : nullptr;   // Z[0] of this instance
        for (int k = 0; k <= N; k++) {
            double z = isx ? x0[k * NS + l] : ((isu && k < N) ? x0[NS * S + k * NC + (l - NS)] : 0.0);
            double xr = xs_l;
            if (TRK) { xr = (k < N && isz) ? zref[(long long)k * NZ + l] : 0.0; row(R_REF, k)[l] = xr; }
            gmax = fmax(gmax, fabs(gradf(k, z, xr)));
            row(R_Z, k)[l] = z;
        }
        gmax = tred_max(gmax);
        this->df = gmax > o.nlp_scaling_max_gradient ? fmax(o.nlp_scaling_max_gradient / gmax, 1e-8) : 1.0;
        double cnt_z = 0.0;
        for (int k = 0; k <= N; k++) {
            double lo = brow(NMPC_BR_BL, k)[l], hi = brow(NMPC_BR_BU, k)[l];
            double z = push_in(row(R_Z, k)[l], lo, hi, o.bound_push, o.bound_frac);
            row(R_Z, k)[l] = z;
            bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
            row(R_ZL, k)[l] = hl ? o.bound_mult_init_val : 0.0;
            row(R_ZU, k)[l] = hu ? o.bound_mult_init_val : 0.0;
            cnt_z += (hl ? 1.0 : 0.0) + (hu ? 1.0 : 0.0);
            row(R_YC, k)[l] = 0.0; row(R_YD, k)[l] = 0.0;
            row(R_CSOC, k)[l] = 0.0; row(R_DSOC, k)[l] = 0.0;
        }
        tsync();
        double cnt_y = isx ? (double)S : 0.0;
        for (int b = 0; b <= N; b++) {
            double s = 0.0, vl = 0.0, vu = 0.0;
            if (isq) {
                double lo = brow(NMPC_BR_DL, b)[l], hi = brow(NMPC_BR_DU, b)[l];
                bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
                double dv = NMPC_DUMMY_ROW_VALUE;
                if (b > 0) dv = rowg(row(R_Z, b - 1), pi, pj, isobs, qob + (b - 1) * qos).dv;
                s = (hl || hu) ? push_in(dv, lo, hi, o.bound_push, o.bound_frac) : dv;
                vl = hl ? o.bound_mult_init_val : 0.0; vu = hu ? o.bound_mult_init_val : 0.0;
                cnt_z += (hl ? 1.0 : 0.0) + (hu ? 1.0 : 0.0);
                cnt_y += (hl || hu) ? 1.0 : 0.0;
            }
            row(R_S, b)[l] = s; row(R_VL, b)[l] = vl; row(R_VU, b)[l] = vu;
        }
        nzb_cnt = tred_sum(cnt_z);
        ny_nzb = tred_sum(cnt_y) + nzb_cnt;
        tsync();
        trig_rows(row, l, N, 0.0, 0, false, R_TRIG);
        this->r_trig = R_TRIG; this->trig_valid = true; this->t2_rdz = -1; this->t2_alpha = 0.0;
    }

    // ---------------------------------------------------------------------------------------
    // residuals / merit quantities at the iterate (FULL) or at a trial point z + alpha dz
    // ---------------------------------------------------------------------------------------
    struct EvalOut { double pinf, viol, dinf, c0, cmu, ysum, zsum, theta, f, slog, sdamp; };

    // cos/sin of every heading of the evaluation point z + alpha dz, all stages at once (one robot-stage per lane per
    // round): row(rt, k)[i] = cos(theta_{i,k}), row(rt, k)[NRP + i] = sin(theta_{i,k}).  Replaces one sincos call per
    // stage in every pass by ceil(N Nr / lanes) calls per evaluation point.
    template <class RowFn>
    static NMPC_DEV void trig_rows(RowFn row, int l, int N, double alpha, int rdz, bool trial, int rt)
    {
        for (int idx = l; idx < N * NR; idx += LW) {
            const int k = idx / NR, i = idx - k * NR;
            double th = row(R_Z, k)[3 * i + 2];
            if (trial) th += alpha * row(rdz, k)[3 * i + 2];
            double s_, c_;
            wp::sincos_(th, &s_, &c_);
            row(rt, k)[i] = c_; row(rt, k)[NRP + i] = s_;
        }
        tsync();
    }

    // Rows of one stage / inequality block, loaded one stage ahead of their use (register software pipeline:
    // the loads of stage k+1 are in flight while stage k is processed, so HBM latency is paid once per pass).
    struct ZRowsB { double z, dz, lo, hi, zl, zu, yc, ce, csoc, cs, sn; };
    struct ZRowsR : ZRowsB { double ref; };   // TRK: with the reference row (a member the other instantiations do not carry)
    typedef typename std::conditional<TRK, ZRowsR, ZRowsB>::type ZRows;
    static NMPC_DEV double zref(const ZRowsR &r) { return r.ref; }
    static NMPC_DEV double zref(const ZRowsB &) { return 0.0; }
    struct QRows { double s, ds, lo, hi, yd, vl, vu, dsoc; };

    // FULL (dual / complementarity terms as well) is a run-time flag: one copy of this pass serves the iterate and the
    // trial points, which halves its instruction-cache footprint
    template <bool FULL>
    NMPC_DEV void eval_pass(double mu, double alpha, int rdz, int rds, bool trial, bool socacc, double asoc, EvalOut &E)
    {
        eval_pass_rt(FULL, mu, alpha, rdz, rds, trial, socacc, asoc, E);
    }
    NMPC_PASS void eval_pass_rt(const bool FULL, double mu, double alpha, int rdz, int rds, bool trial, bool socacc, double asoc, EvalOut &E)
    {
        NMPC_LOCALS
        const double kd = P.o.kappa_d;
        double pinf = 0, viol = 0, dinf = 0, c0 = 0, cmu = 0, ysum = 0, zsum = 0, th = 0, fo = 0, sdamp = 0;
        double *zb = sm + SM_ZB, *ycb = sm + SM_RCB, *ydb = sm + SM_HB;   // (the factorisation's buffers are free during this pass)
        // sum of log(slack) kept as (product of mantissas, sum of exponents): one log() per lane per pass
        double lmant = 1.0;
        int lexp = 0;
        double sprod = 1.0;   // product of this stage's (<= 4) slacks; folded into (mantissa, exponent) once per stage
        auto addlog = [&](double x) { sprod *= x; };
        auto foldlog = [&]() { int e; lmant = wp::frexp_(lmant * sprod, &e); lexp += e; sprod = 1.0; };
        const int rt = trial ? (this->r_trig == R_TRIG ? R_TRIG2 : R_TRIG) : this->r_trig;
        if (trial) { trig_rows(row, l, N, alpha, rdz, true, rt); this->t2_rdz = rdz; this->t2_alpha = alpha; }
        else if (!this->trig_valid) { trig_rows(row, l, N, 0.0, 0, false, rt); this->trig_valid = true; }
        auto load_z = [&](int k) {
            ZRows r;
            k = k < N ? k : N;
            r.cs = row(rt, k < N ? k : N - 1)[rob]; r.sn = row(rt, k < N ? k : N - 1)[NRP + rob];
            r.z = row(R_Z, k)[l]; r.dz = trial ? row(rdz, k)[l] : 0.0;
            r.lo = brow(NMPC_BR_BL, k)[l]; r.hi = brow(NMPC_BR_BU, k)[l]; r.ce = brow(NMPC_BR_CE, k)[l];
            r.zl = FULL ? row(R_ZL, k)[l] : 0.0; r.zu = FULL ? row(R_ZU, k)[l] : 0.0; r.yc = FULL ? row(R_YC, k)[l] : 0.0;
            r.csoc = socacc ? row(R_CSOC, k)[l] : 0.0;
            if constexpr (TRK) r.ref = row(R_REF, k)[l];
            return r;
        };
        auto load_q = [&](int b) {
            QRows r;
            b = b < N ? b : N;
            r.s = row(R_S, b)[l]; r.ds = trial ? row(rds, b)[l] : 0.0;
            r.lo = brow(NMPC_BR_DL, b)[l]; r.hi = brow(NMPC_BR_DU, b)[l];
            r.yd = FULL ? row(R_YD, b)[l] : 0.0; r.vl = FULL ? row(R_VL, b)[l] : 0.0; r.vu = FULL ? row(R_VU, b)[l] : 0.0;
            r.dsoc = socacc ? row(R_DSOC, b)[l] : 0.0;
            return r;
        };
        // one inequality row: residual, merit and (FULL) dual / complementarity terms
        auto ineq_row = [&](int b, const QRows &q, double dv) {
            const bool hl = q.lo > -NMPC_INF, hu = q.hi < NMPC_INF;
            if (!(hl || hu)) return;
            const double s = q.s + alpha * q.ds, dms = dv - s;
            pinf = fmax(pinf, fabs(dms)); th += fabs(dms);
            viol = fmax(viol, fmax(q.lo - dv, dv - q.hi));
            if (socacc) row(R_DSOC, b)[l] = asoc * q.dsoc + dms;
            if (hl) addlog(s - q.lo);
            if (hu) addlog(q.hi - s);
            if (hl && !hu) sdamp += s - q.lo;
            if (hu && !hl) sdamp += q.hi - s;
            if (FULL) {
                ysum += fabs(q.yd);
                double t = -q.yd - q.vl + q.vu;
                if (hl && !hu) t += kd * mu;
                if (hu && !hl) t -= kd * mu;
                dinf = fmax(dinf, fabs(t));
                if (hl) { double u = (s - q.lo) * q.vl; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(q.vl); }
                if (hu) { double u = (q.hi - s) * q.vu; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(q.vu); }
            }
        };
        ZRows zc = load_z(0), zn = load_z(1);
        QRows qn = load_q(1);
        if (isq) { QRows q0 = load_q(0); ineq_row(0, q0, NMPC_DUMMY_ROW_VALUE); }   // block 0: the dummy rows
        for (int k = 0; k <= N; k++) {
            const ZRows zf = load_z(k + 2);          // in flight during this stage
            const QRows qf = load_q(k + 2);
            const bool zv = zvalid(k);
            const double zk = zv ? zc.z + alpha * zc.dz : 0.0;
            zb[l] = zk;
            if (FULL) { ycb[l] = zn.yc; ydb[l] = qn.yd; }   // multipliers of block k+1, read by the other lanes' stationarity rows
            tsync();
            const double csr = zc.cs, snr = zc.sn;   // cos/sin of this lane's robot at stage k
            // ---- equality rows: block 0 (k == 0) and block k+1 ----
            if (isx) {
                if (k == 0) {
                    double c = zk - x0bar_l - zc.ce;
                    pinf = fmax(pinf, fabs(c)); th += fabs(c); viol = fmax(viol, fabs(c));
                    if (socacc) row(R_CSOC, 0)[l] = asoc * zc.csoc + c;
                }
                if (k < N) {
                    double znx = zn.z + alpha * zn.dz;
                    double v = zb[NS + 2 * rob];
                    double pred = comp == 0 ? zk + T * v * csr : (comp == 1 ? zk + T * v * snr : zk + T * zb[NS + 2 * rob + 1]);
                    double c = znx - pred - zn.ce;
                    pinf = fmax(pinf, fabs(c)); th += fabs(c); viol = fmax(viol, fabs(c));
                    if (socacc) row(R_CSOC, k + 1)[l] = asoc * zn.csoc + c;
                }
                if (FULL) ysum += fabs(zc.yc);
            }
            // ---- inequality block k+1 (distances on X_k) ----
            if (isq && k < N) ineq_row(k + 1, qn, rowg(zb, pi, pj, isobs, qob + k * qos).dv);
            // ---- variable bounds, objective, stationarity of stage k ----
            if (zv) {
                const double lo = zc.lo, hi = zc.hi;
                bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
                if (hl) addlog(zk - lo);
                if (hu) addlog(hi - zk);
                if (hl && !hu) sdamp += zk - lo;
                if (hu && !hl) sdamp += hi - zk;
                const double xr = TRK ? zref(zc) : xs_l;
                if (k < N) { double e = zk - xr; fo += 0.5 * qw * e * e; }
                if (FULL) {
                    const double zl = zc.zl, zu = zc.zu;
                    double r = df * gradf(k, zk, xr) - zl + zu;
                    if (hl && !hu) r += kd * mu;
                    if (hu && !hl) r -= kd * mu;
                    if (isx) r += zc.yc;
                    if (k < N) {
                        const double *ycn = ycb;
                        if (isx) {
                            if (comp == 2) {
                                double v = zb[NS + 2 * rob];
                                r -= zn.yc + (-T * v * snr) * ycn[3 * rob] + (T * v * csr) * ycn[3 * rob + 1];
                            } else {
                                r -= zn.yc;
                                const double *ydn = ydb;
                                if (M > 0) {
                                    NMPC_NOUNROLL
                                    for (int j = 0; j < NR; j++) {
                                        if (j == rob) continue;
                                        int q = rob < j ? pairidx(rob, j) : pairidx(j, rob);
                                        r += 2.0 * (zk - zb[3 * j + comp]) * ydn[q];
                                    }
                                }
                                NMPC_NOUNROLL
                                for (int o = 0; o < nobs; o++) {   // this robot's obstacles: gradient (dx, dy) / rho
                                    const double *ob = wp::global_ptr(this->qtab) + k * qos + 3 * o;
                                    const double dx = zb[3 * rob] - ob[0], dy = zb[3 * rob + 1] - ob[1];
                                    r += (comp == 0 ? dx : dy) / sqrt(dx * dx + dy * dy) * ydn[M + rob * nobs + o];
                                }
                            }
                        } else {
                            if (comp == 0) r -= T * (csr * ycn[3 * rob] + snr * ycn[3 * rob + 1]);
                            else r -= T * ycn[3 * rob + 2];
                        }
                    }
                    dinf = fmax(dinf, fabs(r));
                    if (hl) { double u = (zk - lo) * zl; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(zl); }
                    if (hu) { double u = (hi - zk) * zu; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(zu); }
                }
            }
            foldlog();
            zc = zn; zn = zf; qn = qf;
            tsync();
        }
        E.pinf = tred_max(pinf); E.theta = tred_sum(th); E.f = tred_sum(fo);
        E.slog = tred_sum(wp::log_(lmant) + 0.6931471805599453 * (double)lexp); E.sdamp = tred_sum(sdamp); E.viol = tred_max(viol);
        if (FULL) {
            E.dinf = tred_max(dinf); E.c0 = tred_max(c0); E.cmu = tred_max(cmu);
            E.ysum = tred_sum(ysum); E.zsum = tred_sum(zsum);
        }
    }

    // ---------------------------------------------------------------------------------------
    // barrier Hessian / gradient pieces of one variable or slack
    //   MODE 0: primal-dual system;  1: least-squares multiplier estimate;  2: restoration
    // ---------------------------------------------------------------------------------------
    template <int MODE>
    static NMPC_DEV void sig_g(double kd, double v, double lo, double hi, double ml, double mu_, double mu, double g0, double &sig, double &g)
    {
        bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
        if (MODE == 1) { sig = 1.0; g = g0 - ml + mu_; return; }
        sig = 0.0; g = MODE == 0 ? g0 : 0.0;
        if (hl) { double r = wp::rcp_pos(v - lo); sig += MODE == 0 ? ml * r : mu * r * r; g -= mu * r; }
        if (hu) { double r = wp::rcp_pos(hi - v); sig += MODE == 0 ? mu_ * r : mu * r * r; g += mu * r; }
        if (MODE == 0) {
            if (hl && !hu) g += kd * mu;
            if (hu && !hl) g -= kd * mu;
        }
    }

    // inequality block b: condensed weights; writes the per-pair rows the forward pass needs.  The caller supplies the
    // block's inputs (from the staging buffer inside the sweep, from global memory for block 0).
    struct QIn { double lo, hi, s, vl, vu, yd, dsoc; };
    template <int MODE, class RowFn>
    static NMPC_DEV void ineq_block(RowFn row, const QIn &in, int l, int pi, int pj, bool isobs, const double *ob, double kd,
                                    int b, double mu, double delta, bool soc, const double *zb, double &pxx, double &pyy, double &pxy,
                                    double &phx, double &phy)
    {
        pxx = pyy = pxy = phx = phy = 0.0;
        double gxq = 0, gyq = 0, rd = 0, Dq = 0, gs = 0;
        const double lo = in.lo, hi = in.hi;
        if (lo > -NMPC_INF || hi < NMPC_INF) {
            double dv = NMPC_DUMMY_ROW_VALUE, hxx = 0, hyy = 0, hxy = 0;
            if (b > 0) {
                const RowG g = rowg(zb, pi, pj, isobs, ob);
                gxq = g.gx; gyq = g.gy; dv = g.dv; hxx = g.hxx; hyy = g.hyy; hxy = g.hxy;
            }
            double s = in.s, sigs;
            sig_g<MODE>(kd, s, lo, hi, in.vl, in.vu, mu, 0.0, sigs, gs);
            rd = MODE == 1 ? 0.0 : (soc ? in.dsoc : dv - s);
            Dq = sigs + delta;
            const double hq = Dq * rd + gs, yq = MODE == 0 ? in.yd : 0.0;   // multiplier times the row's own curvature
            pxx = Dq * gxq * gxq + yq * hxx; pyy = Dq * gyq * gyq + yq * hyy; pxy = Dq * gxq * gyq + yq * hxy;
            phx = gxq * hq; phy = gyq * hq;
        }
        row(R_GXQ, b)[l] = gxq; row(R_GYQ, b)[l] = gyq; row(R_RD, b)[l] = rd; row(R_DQ, b)[l] = Dq; row(R_GS, b)[l] = gs;
    }

    // ---------------------------------------------------------------------------------------
    // backward Riccati sweep (K3).  false = a control-block pivot was <= 0 (wrong inertia).
    //
    // Lane l < 5Nr holds column l of the stage KKT matrix M = H + [A B]' P+ [A B]: its 3Nr state
    // rows in X[] and its 2Nr control rows in U[]; the last lane holds the linear term m as one more
    // column.  The control block is eliminated by 2Nr symmetric sweeps inside a ROLLED loop: the
    // pivot row is always U[0] (published through shared memory), and the control rows rotate by
    // one register per step (the rotation is folded into the destination registers of the
    // update, so it costs nothing).  A control column's state rows stay 0 until its own pivot
    // (they equal the pivot row by symmetry), which makes the own-column update the same FMA.
    // After the loop X[] holds P (state lanes), K' (control lanes) and p (last lane); U[] of the last
    // lane holds the feed-forward term.
    //
    // The column is assembled directly in the registers by a loop over the robots that is unrolled at compile time:
    // robot i contributes the rows 3i..3i+2 and the control rows 2i, 2i+1 of W = P+ [A B](:, l) (unicycle-sparse: three
    // terms per entry).  Everything else that has to be added to the column -- the collision curvature (x / y lanes), the
    // theta-v cross term, the control diagonal, and, for the last lane, the whole stage gradient h -- arrives as the ADDEND of
    // those FMAs: lane l reads it from five per-lane rows a0p..a4p of small shared-memory tables (x / y / theta rows of robot
    // i, v / omega rows of robot i), so the assembly has no lane-dependent control flow and no register indexing:
    //   x lane of robot r:  a0p = Txx[r], a1p = Txy[r]     Txx[r][j] = -pxx(r,j), Txx[r][r] = +sum_j pxx(r,j)   (same for Tyy, Txy)
    //   y lane of robot r:  a0p = Txy[r], a1p = Tyy[r]
    //   theta lane:         a3p = D3[r]   (crs_r at [r], zeros elsewhere);   v lane: a3p = Dv[r] (its diagonal);   omega lane: a4p = Dw[r]
    //   last lane:          a0p..a4p = HH[0..4]  (the gradient, one row per component class);   every other row: zeros.
    // (The first version built the column through a [5Nr][32] shared-memory column buffer with rolled loops over robots and
    // pairs: 7.7 KB per instance and ~570 instructions per stage, against ~200 and 2.6 KB here.)
    // MODE 3 (sensitivity(), never called by the solve): the matrix of MODE 0 with the stage gradient read from the R_GX rows
    // (a seed) instead of the cost's gradient; with mu = 0 and soc the right-hand side is entirely what the caller put in R_GX,
    // R_CSOC and R_DSOC.
    // ---------------------------------------------------------------------------------------
    template <int MODE>
    NMPC_PASS bool factor(double mu, double delta, bool soc)
    {
        NMPC_LOCALS
        constexpr int MB = MODE == 3 ? 0 : MODE;   // the mode that defines the matrix
        const double zeta = MODE == 2 ? sqrt(mu) : 0.0, kd = this->P.o.kappa_d;
        const bool isL = (l == LW - 1);
        double X[NS], U[NC];
        double plin = 0.0, dgx = 0.0;
        double *col = sm + SM_COL, *pb = sm + SM_PB, *zb = sm + SM_ZB, *rcb = sm + SM_RCB, *prb = sm + SM_PRB, *hb = sm + SM_HB;
        double *cs = sm + SM_CS, *sn = sm + SM_SN, *c4 = sm + SM_C4, *crs = sm + SM_CRS, *thd = sm + SM_THD;
        double *tt = sm + SM_TT, *HH = tt + 8 * TSZ, *ZR = HH + 5 * NR;
        double *stg = sm + SM_STG;
        n_fact++;
        tsync();
        // the big region was the forward pass's staging buffer: reset the constant zeros of the addend tables and of the two
        // padding columns of the P buffer (the last lane multiplies them by 0)
        for (int e = l; e < 8 * TSZ + 6 * NR; e += LW) tt[e] = 0.0;
        for (int e = l; e < NS; e += LW) { pb[e * PLD + NS + 1] = 0.0; pb[e * PLD + NS + 2] = 0.0; }
        // addend rows of this lane (see above), the diagonal entry this lane maintains, and this lane's row-sum job
        const double *a0p = ZR, *a1p = ZR, *a2p = ZR, *a3p = ZR, *a4p = ZR;
        double *selfp = nullptr;         // diagonal entry of D3 / Dv / Dw owned by this lane
        double *hslot = nullptr;         // where this lane's stage gradient goes (HH)
        if (isx) {
            hslot = HH + comp * NR + rob;
            if (comp == 0) { a0p = tt + 0 * TSZ + rob * TCOLS; a1p = tt + 1 * TSZ + rob * TCOLS; }
            else if (comp == 1) { a0p = tt + 1 * TSZ + rob * TCOLS; a1p = tt + 2 * TSZ + rob * TCOLS; }
            else { a3p = tt + 5 * TSZ + rob * TCOLS; selfp = tt + 5 * TSZ + rob * (TCOLS + 1); }
        } else if (isu) {
            hslot = HH + (3 + comp) * NR + rob;
            if (comp == 0) { a3p = tt + 6 * TSZ + rob * TCOLS; selfp = tt + 6 * TSZ + rob * (TCOLS + 1); }
            else { a4p = tt + 7 * TSZ + rob * TCOLS; selfp = tt + 7 * TSZ + rob * (TCOLS + 1); }
        } else if (isL) { a0p = HH; a1p = HH + NR; a2p = HH + 2 * NR; a3p = HH + 3 * NR; a4p = HH + 4 * NR; }
        // row sums of the five pair tables: lane a * NR + i sums row i of table a and stores it on the diagonal
        const bool rsum_any = M > 0 || nobs > 0, rsum = rsum_any && l < 5 * NR;
        const int rs_a = l / NR, rs_i = l - rs_a * NR, rs_n = NR + nobs;
        double *rs_row = tt + rs_a * TSZ + rs_i * TCOLS;
        // column l of [A B]:  al e_x + be e_y + ga e_theta of this lane's robot (last lane: the pr column); xm: control lanes keep
        // their state rows at 0 until their own pivot (see the sweep)
        const double xm = isu ? 0.0 : 1.0;
        const int base = isL ? NS : 3 * rob;
        tsync();
        // staging of stage k: four contiguous ranges (see FS_*)
        double *const bar = sm + SM_MBAR;
        auto stage_issue = [&](int k) {
            if (l == 0) {
                wp::fence_proxy_async();
                wp::bulk_expect(bar, (unsigned)(FS_COUNT * LW * sizeof(double)));
                bulk_rows(bar, stg + FS_REF * LW, row(R_REF, k), FS_BL - FS_REF);
                bulk_rows(bar, stg + FS_BL * LW, brow(NMPC_BR_BL, k), 2);
                bulk_rows(bar, stg + FS_YC * LW, row(R_YC, k + 1), FS_CE - FS_YC);
                bulk_rows(bar, stg + FS_CE * LW, brow(NMPC_BR_CE, k + 1), 3);
            }
        };
        const int fs_trig = FS_TRIG2 + (this->r_trig - R_TRIG2);   // which of the two trig rows belongs to the iterate
        stage_issue(N - 1);   // in flight during the terminal stage
        // terminal stage: X_N carries no cost and no distance rows, only its box
        {
            double sig = 0.0, gx = 0.0;
            if (isx) sig_g<MB>(kd, row(R_Z, N)[l], brow(NMPC_BR_BL, N)[l], brow(NMPC_BR_BU, N)[l], row(R_ZL, N)[l], row(R_ZU, N)[l], mu,
                               MODE == 3 ? row(R_GX, N)[l] : 0.0, sig, gx);
            hb[l] = isx ? gx : 0.0;
            tsync();
            NMPC_UNROLL
            for (int i = 0; i < NS; i++) X[i] = isL ? hb[i] : 0.0;
            dgx = isx ? sig + delta + zeta : 0.0;   // P_N = X + diag(dgx): the own-row diagonal is carried separately
            NMPC_UNROLL
            for (int u = 0; u < NC; u++) U[u] = 0.0;
            plin = isx ? gx : 0.0;
            row(R_GX, N)[l] = plin;
            NMPC_UNROLL
            for (int i = 0; i < NS; i++) frow(N, i)[l] = isz ? X[i] : 0.0;
            row(R_LIN, N)[l] = plin; row(R_DG, N)[l] = dgx;
            zb[l] = isx ? row(R_Z, N)[l] : 0.0;   // read back by the same lane as X_{k+1} of the first stage
        }
        NMPC_NOUNROLL
        for (int k = N - 1; k >= 0; k--) {
            stage_wait();
            tsync();
            const double zk = isz ? stg[FS_Z * LW + l] : 0.0;
            const double znx = zb[l];   // X_{k+1} (this lane's component): what the previous stage left here
            zb[l] = zk;
            if (l < NR) {
                const double *zr = stg + FS_Z * LW;
                const double v = zr[NS + 2 * l], c_ = stg[fs_trig * LW + l], s_ = stg[fs_trig * LW + NRP + l];
                cs[l] = c_; sn[l] = s_;
                double a_ = -T * v * s_, b_ = T * v * c_, tc = T * c_, ts = T * s_;
                c4[4 * l] = a_; c4[4 * l + 1] = b_; c4[4 * l + 2] = tc; c4[4 * l + 3] = ts;
                double *cf = row(R_COEF, k);
                cf[l] = a_; cf[CFS + l] = b_; cf[2 * CFS + l] = tc; cf[3 * CFS + l] = ts;
                if (MB == 0) {
                    const double *yc = stg + FS_YC * LW;
                    double lx = yc[3 * l], ly = yc[3 * l + 1];
                    crs[l] = T * (lx * s_ - ly * c_); thd[l] = T * v * (lx * c_ + ly * s_);
                } else { crs[l] = 0.0; thd[l] = 0.0; }
            }
            if (isx) {
                NMPC_UNROLL
                for (int i = 0; i < NS; i++) pb[i * PLD + l] = X[i];
                pb[l * PLD + l] += dgx;   // same lane wrote this element just above
            }
            if (rsum) rs_row[rs_i] = 0.0;   // the diagonal is summed over below: clear the previous stage's sum
            tsync();
            // equality residual of block k+1 and the condensed inequality block k+1
            if (isx) {
                double rc = 0.0;
                if (MODE != 1) {
                    if (soc) rc = stg[FS_CSOC * LW + l];
                    else {
                        double v = zb[NS + 2 * rob];
                        double pred = comp == 0 ? zk + T * v * cs[rob] : (comp == 1 ? zk + T * v * sn[rob] : zk + T * zb[NS + 2 * rob + 1]);
                        rc = znx - pred - stg[FS_CE * LW + l];
                    }
                }
                rcb[l] = rc; row(R_RC, k + 1)[l] = rc;
            }
            if (isq) {
                double a0, a1, a2, a3, a4;
                QIn in;
                in.lo = stg[FS_DL * LW + l]; in.hi = stg[FS_DU * LW + l]; in.s = stg[FS_S * LW + l]; in.vl = stg[FS_VL * LW + l];
                in.vu = stg[FS_VU * LW + l]; in.yd = stg[FS_YD * LW + l]; in.dsoc = stg[FS_DSOC * LW + l];
                ineq_block<MB>(row, in, l, pi, pj, isobs, qob + k * qos, kd, k + 1, mu, delta, soc, zb, a0, a1, a2, a3, a4);
                // pair row: entries (pi, pj) and (pj, pi); obstacle row: column NR + o of robot pi (it only feeds the row sum)
                const int e1 = isobs ? pi * TCOLS + NR + (l - M) % nobs : pi * TCOLS + pj, e2 = isobs ? e1 : pj * TCOLS + pi;
                tt[e2] = -a0; tt[TSZ + e2] = -a2; tt[2 * TSZ + e2] = -a1; tt[3 * TSZ + e2] = -a3; tt[4 * TSZ + e2] = -a4;
                tt[e1] = -a0;                                                 // Txx
                tt[TSZ + e1] = -a2;                                           // Txy
                tt[2 * TSZ + e1] = -a1;                                       // Tyy
                tt[3 * TSZ + e1] = a3;                                        // Thx: gradient of robot pi gets +, of robot pj gets -
                tt[4 * TSZ + e1] = a4;                                        // Thy
            }
            tsync();
            // pr = p_{k+1} + P_{k+1} r (r = -rc), published as one more column of pb for the last lane
            if (isx) {
                double pr = plin;
                if (MODE != 1) {
                    NMPC_UNROLL
                    for (int i = 0; i < NS; i++) pr -= X[i] * rcb[i];
                    pr -= dgx * rcb[l];
                }
                pb[l * PLD + NS] = pr;
            }
            if (rsum) {   // diagonal of the curvature tables = + sum of the pair terms; of the gradient tables = the robot's sum
                double s_ = 0.0;
                if (NOBS_MAX == 0 || nobs == 0) {
                    NMPC_UNROLL
                    for (int j = 0; j < NR; j++) s_ += rs_row[j];
                } else {
                    for (int j = 0; j < rs_n; j++) s_ += rs_row[j];
                }
                rs_row[rs_i] = rs_a < 3 ? -s_ : s_;
            }
            // stage gradient h_l (variable l) and diagonal curvature
            double sig = 0.0, gx = 0.0, dg = 0.0;
            if (isz) {
                sig_g<MB>(kd, zk, stg[FS_BL * LW + l], stg[FS_BU * LW + l], stg[FS_ZL * LW + l], stg[FS_ZU * LW + l], mu,
                          MODE == 3 ? row(R_GX, k)[l] : df * gradf(k, zk, TRK ? stg[FS_REF * LW + l] : xs_l), sig, gx);
                dg = sig + delta + zeta;
                if (MB == 0) { dg += df * qw; if (isx && comp == 2) dg += thd[rob]; }
            }
            row(R_GX, k)[l] = gx;
            dgx = isx ? dg : 0.0;                                                   // state diagonal is carried lazily
            if (selfp) *selfp = isu ? dg : (MB == 0 ? crs[rob] : 0.0);           // control diagonal / theta-v cross term
            tsync();
            if (isz) *hslot = gx + ((rsum_any && isx && comp < 2) ? tt[(3 + comp) * TSZ + rob * (TCOLS + 1)] : 0.0);
            tsync();
            if (k > 0) stage_issue(k - 1);   // every lane has consumed the staged rows of stage k
            {
                const double al = isL ? 1.0 : (isx ? (comp == 0 ? 1.0 : (comp == 2 ? c4[4 * rob] : 0.0)) : (isu && comp == 0 ? c4[4 * rob + 2] : 0.0));
                const double be = isx ? (comp == 1 ? 1.0 : (comp == 2 ? c4[4 * rob + 1] : 0.0)) : (isu && comp == 0 ? c4[4 * rob + 3] : 0.0);
                const double ga = isx ? (comp == 2 ? 1.0 : 0.0) : (isu && comp == 1 ? T : 0.0);
                const double *pbl = pb + base;
                NMPC_UNROLL
                for (int i = 0; i < NR; i++) {
                    const double *q0 = pbl + (3 * i) * PLD;
                    const double Wx = al * q0[0] + be * q0[1] + ga * q0[2];
                    const double Wy = al * q0[PLD] + be * q0[PLD + 1] + ga * q0[PLD + 2];
                    const double Wt = al * q0[2 * PLD] + be * q0[2 * PLD + 1] + ga * q0[2 * PLD + 2];
                    const double ca_ = c4[4 * i], cb_ = c4[4 * i + 1], tc_ = c4[4 * i + 2], ts_ = c4[4 * i + 3];
                    X[3 * i] = fma(xm, Wx, a0p[i]);
                    X[3 * i + 1] = fma(xm, Wy, a1p[i]);
                    X[3 * i + 2] = fma(xm, fma(ca_, Wx, fma(cb_, Wy, Wt)), a2p[i]);
                    U[2 * i] = fma(tc_, Wx, fma(ts_, Wy, a3p[i]));
                    U[2 * i + 1] = fma(T, Wt, a4p[i]);
                }
            }
            // symmetric sweep of the control pivots (rolled, with one-pivot LOOK-AHEAD).  The pivot row is U[0] of
            // every lane; it is published in ROTATED order (slot NS + r holds control column (j + r) mod 2Nr), so the
            // readers use compile-time offsets and the rows rotate through the registers for free.  A second row of
            // the buffer carries 1/entry, so 1/pivot comes from the pivot's own lane (<= 0, inf or NaN: wrong inertia).  Inside step j the entry of
            // the NEXT pivot row is updated and published first, so its shared-memory round trip and reciprocal
            // overlap the remaining rank-1 update instead of sitting on the critical path of every pivot.
            const int ucol = l - NS;   // control column of this lane (if any)
            int pslot = l;             // where this lane publishes its entry of the next pivot row (control lanes: rotating)
            col[pslot] = U[0]; col[LW + pslot] = wp::rcp_pos(U[0]);   // every lane (no branch): the slots of the lanes beyond the 5Nr columns are never read
            // one pivot step; the loop below is unrolled by two so that both buffers have compile-time addresses
            auto pivot = [&](const int j, const double *buf, double *nbuf) -> bool {
                tsync();
                const double inv = buf[LW + NS];   // 1 / pivot, from the pivot's own lane (rotated slot NS)
                if (!wp::pos_normal(inv)) return false;
                // the control part of the pivot row first (128-bit loads): it feeds the look-ahead
                double bu[NC];
                if ((NS & 1) == 0) {
                    const NmpcD2 *c2 = reinterpret_cast<const NmpcD2 *>(buf + NS);
                    NMPC_UNROLL
                    for (int r = 0; r < NC / 2; r++) { NmpcD2 v = c2[r]; bu[2 * r] = v.x; bu[2 * r + 1] = v.y; }
                } else {
                    NMPC_UNROLL
                    for (int r = 0; r < NC; r++) bu[r] = buf[NS + r];
                }
                const bool own = (ucol == j);
                const double t = own ? -inv : U[0] * inv;
                const double tx = (ucol > j && isu) ? 0.0 : t;
                if (own) {   // the pivot column becomes column / d: start its remaining rows from 0.  (Predicated moves instead of
                             // this divergent branch were measured: 22 FSEL in front of the FMAs, 45.2 k -> 42.0 k solves/s.)
                    NMPC_UNROLL
                    for (int r = 1; r < NC; r++) U[r] = 0.0;
                }
                // look-ahead: this lane's entry of pivot row j+1 (the publish after the last pivot is harmless: that buffer is not read again)
                const double u1 = U[1] - bu[1] * t;
                if (isu) { pslot--; pslot += pslot < NS ? NC : 0; }
                const double r1 = wp::rcp_pos(u1);   // every lane: no divergent reciprocal
                nbuf[pslot] = u1; nbuf[LW + pslot] = r1;
                // control rows (rotating): slots NS+2 .. NS+NC-1
                U[0] = u1;
                NMPC_UNROLL
                for (int r = 2; r < NC; r++) U[r - 1] = U[r] - bu[r] * t;
                U[NC - 1] = t;
                // state rows in batches of XB pairs, each batch loaded while the previous one is consumed: the whole pivot row
                // in registers at once (the first version) costs 60 registers and caps the kernel at 12 warps per SM
                {
                    constexpr int NP = NS / 2, XB = NMPC_XBATCH;
                    const NmpcD2 *b2 = reinterpret_cast<const NmpcD2 *>(buf);
                    NmpcD2 cur[XB], nxt[XB];
                    NMPC_UNROLL
                    for (int i = 0; i < XB; i++) if (i < NP) cur[i] = b2[i];
                    NMPC_UNROLL
                    for (int i0 = 0; i0 < NP; i0 += XB) {
                        NMPC_UNROLL
                        for (int i = 0; i < XB; i++) if (i0 + XB + i < NP) nxt[i] = b2[i0 + XB + i];
                        wp::sched_fence();
                        NMPC_UNROLL
                        for (int i = 0; i < XB; i++)
                            if (i0 + i < NP) { X[2 * (i0 + i)] -= cur[i].x * tx; X[2 * (i0 + i) + 1] -= cur[i].y * tx; }
                        NMPC_UNROLL
                        for (int i = 0; i < XB; i++) cur[i] = nxt[i];
                    }
                    if (NS & 1) X[NS - 1] -= buf[NS - 1] * tx;
                }
                return true;
            };
#if NMPC_PIVOT_UNROLL == 2
            NMPC_NOUNROLL
            for (int j = 0; j < NC; j += 2) {
                if (!pivot(j, col, col + 2 * LW) || !pivot(j + 1, col + 2 * LW, col)) { if (k > 0) stage_wait(); return false; }   // drain the staging copy in flight before the retry
            }
#else
            NMPC_NOUNROLL
            for (int j = 0; j < NC; j++) {
                if (!pivot(j, col + 2 * LW * (j & 1), col + 2 * LW * ((j + 1) & 1))) { if (k > 0) stage_wait(); return false; }   // drain the staging copy in flight before the retry
            }
#endif
            // publish p_k / feed-forward (the last lane's column) and store the factors
            tsync();
            if (isL) {
                NMPC_UNROLL
                for (int i = 0; i < NS; i++) prb[i] = X[i];
                NMPC_UNROLL
                for (int u = 0; u < NC; u++) prb[NS + u] = U[u];
            }
            tsync();
            if (isz) {
                const double v = prb[l];
                plin = v;
                row(R_LIN, k)[l] = v; row(R_DG, k)[l] = dgx;
                double *fp = frow(k, 0) + l;   // one address, compile-time row offsets
                NMPC_UNROLL
                for (int i = 0; i < NS; i++) fp[i * LW] = X[i];
            }
        }
        tsync();
        if (isx) row(R_RC, 0)[l] = MODE == 1 ? 0.0 : (soc ? row(R_CSOC, 0)[l] : row(R_Z, 0)[l] - x0bar_l - brow(NMPC_BR_CE, 0)[l]);
        if (isq) {
            double a0, a1, a2, a3, a4;
            QIn in;
            in.lo = brow(NMPC_BR_DL, 0)[l]; in.hi = brow(NMPC_BR_DU, 0)[l]; in.s = row(R_S, 0)[l]; in.vl = row(R_VL, 0)[l]; in.vu = row(R_VU, 0)[l];
            in.yd = MB == 0 ? row(R_YD, 0)[l] : 0.0; in.dsoc = soc ? row(R_DSOC, 0)[l] : 0.0;
            ineq_block<MB>(row, in, l, pi, pj, isobs, qob, kd, 0, mu, delta, soc, zb, a0, a1, a2, a3, a4);
        }
        tsync();
        return true;
    }

    // ---------------------------------------------------------------------------------------
    // forward pass: steps, new multipliers, fraction-to-boundary step sizes, grad(phi)'d
    // ---------------------------------------------------------------------------------------
    struct StepInfo { double ap, az, gbd, tiny; };

    // fraction-to-boundary bookkeeping of one bounded quantity: rp = max(-dv/slack), rz = max(-dmult/mult);
    // the step sizes are tau / max ratio (one division per pass instead of one per bound)
    static NMPC_DEV void slack_step_terms(double v, double dv, double lo, double hi, double ml, double mu_, double mu, double &rp,
                                          double &rz)
    {
        if (lo > -NMPC_INF) {
            double r = wp::rcp_pos(v - lo);
            rp = fmax(rp, -dv * r);
            double dm = mu * r - ml - ml * r * dv;
            rz = fmax(rz, -dm * wp::rcp_pos(ml));
        }
        if (hi < NMPC_INF) {
            double r = wp::rcp_pos(hi - v);
            rp = fmax(rp, dv * r);
            double dm = mu * r - mu_ + mu_ * r * dv;
            rz = fmax(rz, -dm * wp::rcp_pos(mu_));
        }
    }

    NMPC_PASS void forward(double mu, double tau, int rdz, int rds, int rytc, int rytd, StepInfo &si)
    {
        NMPC_LOCALS
        double ap = 0.0, az = 0.0, gbd = 0.0, tiny = 0.0;   // max ratios, see slack_step_terms
        double *dzb = sm + SM_DZB;
        double *stg = sm + SM_BIG;  // the factorisation's buffers are free during this pass: WS_COUNT staging rows
        double *const bar = sm + SM_MBAR;
        tsync();
        // staging of stage k: four contiguous ranges (see WS_*); block k + 1 clamped to N
        auto issue = [&](int k) {
            const int kb = k < N ? k + 1 : N;
            if (l == 0) {
                wp::fence_proxy_async();
                wp::bulk_expect(bar, (unsigned)(WS_COUNT * LW * sizeof(double)));
                bulk_rows(bar, stg + WS_Z * LW, row(R_Z, k), WS_BL - WS_Z);
                bulk_rows(bar, stg + WS_BL * LW, brow(NMPC_BR_BL, k), 2);
                bulk_rows(bar, stg + WS_S * LW, row(R_S, kb), WS_DL - WS_S);
                bulk_rows(bar, stg + WS_DL * LW, brow(NMPC_BR_DL, kb), 2);
            }
        };
        issue(0);
        double dx = isx ? -row(R_RC, 0)[l] : 0.0;
        if (isq) {
            double rd = row(R_RD, 0)[l], Dq = row(R_DQ, 0)[l], gs = row(R_GS, 0)[l];
            bool act = brow(NMPC_BR_DL, 0)[l] > -NMPC_INF || brow(NMPC_BR_DU, 0)[l] < NMPC_INF;
            double ds = act ? rd : 0.0, ytd = act ? Dq * ds + gs : 0.0;
            row(rds, 0)[l] = ds; row(rytd, 0)[l] = ytd;
            if (act) {
                double s = row(R_S, 0)[l];
                slack_step_terms(s, ds, brow(NMPC_BR_DL, 0)[l], brow(NMPC_BR_DU, 0)[l], row(R_VL, 0)[l], row(R_VU, 0)[l], mu, ap, az);
                gbd += gs * ds; tiny = fmax(tiny, fabs(ds) / (1.0 + fabs(s)));
            }
        }
        for (int k = 0; k <= N; k++) {
            stage_wait();
            if (isx) dzb[l] = dx;
            tsync();
            // everything this stage needs moves from the staging buffer to registers, then the buffer is refilled
            // for stage k+1 while this stage computes
            double fv[NS];
            NMPC_UNROLL
            for (int i = 0; i < NS; i++) fv[i] = stg[(WS_F0 + i) * LW + l];
            const double v_lin = stg[WS_LIN * LW + l], v_dg = stg[WS_DG * LW + l], v_z = stg[WS_Z * LW + l], v_zl = stg[WS_ZL * LW + l],
                         v_zu = stg[WS_ZU * LW + l], v_bl = stg[WS_BL * LW + l], v_bu = stg[WS_BU * LW + l], v_gx = stg[WS_GX * LW + l];
            const double *cf = stg + WS_COEF * LW;
            const double cA = comp == 0 ? cf[rob] : (comp == 1 ? cf[CFS + rob] : 0.0);
            const double cB = comp == 0 ? cf[2 * CFS + rob] : (comp == 1 ? cf[3 * CFS + rob] : T);
            const double v_rc = stg[WS_RC * LW + l];
            const double q_lo = stg[WS_DL * LW + l], q_hi = stg[WS_DU * LW + l], q_gs = stg[WS_GS * LW + l], q_gx = stg[WS_GXQ * LW + l],
                         q_gy = stg[WS_GYQ * LW + l], q_rd = stg[WS_RD * LW + l], q_dq = stg[WS_DQ * LW + l], q_s = stg[WS_S * LW + l],
                         q_vl = stg[WS_VL * LW + l], q_vu = stg[WS_VU * LW + l];
            tsync();
            if (k < N) issue(k + 1);
            double acc = 0.0;
            if (isz) {
                double a0 = v_lin, a1 = isx ? v_dg * dzb[l] : 0.0, a2 = 0.0;
                NMPC_UNROLL
                for (int i = 0; i < NS; i += 3) {   // three accumulation chains
                    a0 += fv[i] * dzb[i];
                    a1 += fv[i + 1] * dzb[i + 1];
                    a2 += fv[i + 2] * dzb[i + 2];
                }
                acc = a0 + (a1 + a2);
            }
            if (isx) row(rytc, k)[l] = -acc;
            const double du = (isu && k < N) ? -acc : 0.0;
            if (isu) dzb[l] = du;
            const double dzl = isx ? dx : du;
            row(rdz, k)[l] = dzl;
            if (zvalid(k)) {
                slack_step_terms(v_z, dzl, v_bl, v_bu, v_zl, v_zu, mu, ap, az);
                gbd += v_gx * dzl; tiny = fmax(tiny, fabs(dzl) / (1.0 + fabs(v_z)));
            }
            if (k < N) {
                tsync();
                double dn = 0.0;
                if (isx) dn = dzb[l] + cA * dzb[3 * rob + 2] + cB * dzb[NS + 2 * rob + (comp == 2 ? 1 : 0)] - v_rc;
                if (isq) {
                    const int b = k + 1;
                    bool act = q_lo > -NMPC_INF || q_hi < NMPC_INF;
                    double ds = 0.0, ytd = 0.0;
                    if (act) {
                        ds = q_gx * (dzb[3 * pi] - (isobs ? 0.0 : dzb[3 * pj])) + q_gy * (dzb[3 * pi + 1] - (isobs ? 0.0 : dzb[3 * pj + 1])) + q_rd;
                        ytd = q_dq * ds + q_gs;
                        slack_step_terms(q_s, ds, q_lo, q_hi, q_vl, q_vu, mu, ap, az);
                        gbd += q_gs * ds; tiny = fmax(tiny, fabs(ds) / (1.0 + fabs(q_s)));
                    }
                    row(rds, b)[l] = ds; row(rytd, b)[l] = ytd;
                }
                dx = dn;
                tsync();   // dzb is rewritten at the top of the next stage
            }
        }
        ap = tred_max(ap); az = tred_max(az);
        si.ap = ap > tau ? tau / ap : 1.0; si.az = az > tau ? tau / az : 1.0;
        si.gbd = tred_sum(gbd); si.tiny = tred_max(tiny);
        tsync();
    }

    // ---------------------------------------------------------------------------------------
    NMPC_PASS void accept(double alpha, double az, double mu, int rdz, int rds, int rytc, int rytd)
    {
        NMPC_LOCALS
        if (this->t2_rdz == rdz && this->t2_alpha == alpha) { this->r_trig = this->r_trig == R_TRIG ? R_TRIG2 : R_TRIG; this->trig_valid = true; }
        else this->trig_valid = false;
        this->t2_rdz = -1;
        const double ks = this->P.o.kappa_sigma, iks = 1.0 / ks;
        // bound multiplier after the step, kept in the kappa_sigma corridor around mu / (new slack)
        auto mult = [=](double m, double sl_old, double sl_new, double dv_signed) {
            double r = wp::rcp_pos(sl_old), c = mu * wp::rcp_pos(sl_new);
            double m2 = m + az * (mu * r - m + m * r * dv_signed);
            return fmax(fmin(m2, ks * c), iks * c);
        };
        struct AR { double z, dz, lo, hi, zl, zu, yc, ytc, s, ds, dlo, dhi, vl, vu, yd, ytd; };
        auto load = [&](int k) {   // all rows of stage / block k, issued together one stage ahead of their use
            AR r;
            k = k < N ? k : N;
            r.z = row(R_Z, k)[l]; r.dz = row(rdz, k)[l]; r.lo = brow(NMPC_BR_BL, k)[l]; r.hi = brow(NMPC_BR_BU, k)[l];
            r.zl = row(R_ZL, k)[l]; r.zu = row(R_ZU, k)[l]; r.yc = row(R_YC, k)[l]; r.ytc = row(rytc, k)[l];
            r.s = row(R_S, k)[l]; r.ds = row(rds, k)[l]; r.dlo = brow(NMPC_BR_DL, k)[l]; r.dhi = brow(NMPC_BR_DU, k)[l];
            r.vl = row(R_VL, k)[l]; r.vu = row(R_VU, k)[l]; r.yd = row(R_YD, k)[l]; r.ytd = row(rytd, k)[l];
            return r;
        };
        AR c = load(0);
        for (int k = 0; k <= N; k++) {
            const AR nx = load(k + 1);
            if (zvalid(k)) {
                const double zn = c.z + alpha * c.dz;
                if (c.lo > -NMPC_INF) row(R_ZL, k)[l] = mult(c.zl, c.z - c.lo, zn - c.lo, -c.dz);
                if (c.hi < NMPC_INF) row(R_ZU, k)[l] = mult(c.zu, c.hi - c.z, c.hi - zn, c.dz);
                row(R_Z, k)[l] = zn;
            }
            if (isx) row(R_YC, k)[l] = c.yc + alpha * (c.ytc - c.yc);
            if (isq && (c.dlo > -NMPC_INF || c.dhi < NMPC_INF)) {
                const double sn_ = c.s + alpha * c.ds;
                if (c.dlo > -NMPC_INF) row(R_VL, k)[l] = mult(c.vl, c.s - c.dlo, sn_ - c.dlo, -c.ds);
                if (c.dhi < NMPC_INF) row(R_VU, k)[l] = mult(c.vu, c.dhi - c.s, c.dhi - sn_, c.ds);
                row(R_S, k)[l] = sn_;
                row(R_YD, k)[l] = c.yd + alpha * (c.ytd - c.yd);
            }
            c = nx;
        }
        tsync();
    }

    NMPC_PASS void accept_primal(double alpha, int rdz, int rds)
    {
        NMPC_LOCALS
        this->trig_valid = false; this->t2_rdz = -1;
        for (int k = 0; k <= N; k++) {
            if (zvalid(k)) row(R_Z, k)[l] += alpha * row(rdz, k)[l];
            if (isq && (brow(NMPC_BR_DL, k)[l] > -NMPC_INF || brow(NMPC_BR_DU, k)[l] < NMPC_INF)) row(R_S, k)[l] += alpha * row(rds, k)[l];
        }
        tsync();
    }

    // after the restoration fallback: equality multipliers reset, bound multipliers clipped
    NMPC_PASS void resto_reset(double mu)
    {
        NMPC_LOCALS
        const double ks = P.o.kappa_sigma;
        for (int k = 0; k <= N; k++) {
            if (zvalid(k)) {
                double z = row(R_Z, k)[l], lo = brow(NMPC_BR_BL, k)[l], hi = brow(NMPC_BR_BU, k)[l];
                if (lo > -NMPC_INF) { double s2 = z - lo; row(R_ZL, k)[l] = fmax(fmin(row(R_ZL, k)[l], ks * mu / s2), mu / (ks * s2)); }
                if (hi < NMPC_INF) { double s2 = hi - z; row(R_ZU, k)[l] = fmax(fmin(row(R_ZU, k)[l], ks * mu / s2), mu / (ks * s2)); }
            }
            row(R_YC, k)[l] = 0.0; row(R_YD, k)[l] = 0.0;
            if (isq) {
                double s = row(R_S, k)[l], lo = brow(NMPC_BR_DL, k)[l], hi = brow(NMPC_BR_DU, k)[l];
                if (lo > -NMPC_INF) { double s2 = s - lo; row(R_VL, k)[l] = fmax(fmin(row(R_VL, k)[l], ks * mu / s2), mu / (ks * s2)); }
                if (hi < NMPC_INF) { double s2 = hi - s; row(R_VU, k)[l] = fmax(fmin(row(R_VU, k)[l], ks * mu / s2), mu / (ks * s2)); }
            }
        }
        tsync();
    }

    // restoration candidate: forward rollout of the current controls (every equality row becomes zero) and
    // slacks reset from the distances; written as a direction (R_DZ, R_DS) = candidate - iterate
    NMPC_PASS void rollout_project()
    {
        NMPC_LOCALS
        const nmpc_opts &o = this->P.o;
        double *zb = sm + SM_ZB, *cs = sm + SM_CS, *sn = sm + SM_SN;
        double zt = isx ? push_in(x0bar_l + brow(NMPC_BR_CE, 0)[l], brow(NMPC_BR_BL, 0)[l], brow(NMPC_BR_BU, 0)[l], o.bound_push, o.bound_frac) : (isu ? row(R_Z, 0)[l] : 0.0);
        for (int k = 0; k <= N; k++) {
            const bool zv = zvalid(k);
            row(R_DZ, k)[l] = zv ? zt - row(R_Z, k)[l] : 0.0;
            zb[l] = zv ? zt : 0.0;
            tsync();
            if (k < N && l < NR) { double s_, c_; wp::sincos_(zb[3 * l + 2], &s_, &c_); cs[l] = c_; sn[l] = s_; }
            if (isq) {
                for (int pass = (k == 0 ? 0 : 1); pass < 2; pass++) {
                    if (pass == 1 && k == N) break;
                    const int b = pass == 0 ? 0 : k + 1;
                    double lo = brow(NMPC_BR_DL, b)[l], hi = brow(NMPC_BR_DU, b)[l], dv = NMPC_DUMMY_ROW_VALUE;
                    if (pass == 1) dv = rowg(zb, pi, pj, isobs, qob + k * qos).dv;
                    bool act = lo > -NMPC_INF || hi < NMPC_INF;
                    row(R_DS, b)[l] = act ? push_in(dv, lo, hi, o.bound_push, o.bound_frac) - row(R_S, b)[l] : 0.0;
                }
            }
            tsync();
            if (k < N) {
                double zn = 0.0;
                if (isx) {
                    double v = zb[NS + 2 * rob];
                    zn = comp == 0 ? zt + T * v * cs[rob] : (comp == 1 ? zt + T * v * sn[rob] : zt + T * zb[NS + 2 * rob + 1]);
                    zn = push_in(zn + brow(NMPC_BR_CE, k + 1)[l], brow(NMPC_BR_BL, k + 1)[l], brow(NMPC_BR_BU, k + 1)[l], o.bound_push, o.bound_frac);
                } else if (isu && k + 1 < N) zn = row(R_Z, k + 1)[l];
                zt = zn;
            }
            tsync();
        }
    }

    // copy the initial-residual rows into the SOC accumulators (c_soc := c, d_soc := d - s)
    NMPC_PASS void soc_begin()
    {
        NMPC_LOCALS
        for (int k = 0; k <= N; k++) {
            row(R_CSOC, k)[l] = isx ? row(R_RC, k)[l] : 0.0;
            row(R_DSOC, k)[l] = (isq) ? row(R_RD, k)[l] : 0.0;
        }
        tsync();
    }

    // ---------------------------------------------------------------------------------------
    // filter.  IPOPT's filter is unbounded inside a barrier subproblem (it is reset when mu changes); the benchmark instances
    // add up to 104 entries to it (oracle, 4,096 instances), so it lives in the per-slot global scratch, append-only:
    // entries that a new one dominates are redundant for the acceptance test and are simply left in place.  Every lane checks
    // its share of the entries.  An overflow of the NMPC_FILTER_CAP entries overwrites the oldest and is counted (stats).
    // ---------------------------------------------------------------------------------------
    NMPC_DEV double *filter_base() const { return ws + (long long)R_COUNT * S * LW; }
    NMPC_DEV bool filter_ok(double th, double ph) const
    {
        const double *fth = wp::global_ptr(filter_base()), *fph = fth + NMPC_FILTER_CAP;
        const int m = fn < NMPC_FILTER_CAP ? fn : NMPC_FILTER_CAP;
        bool ok = true;
        for (int i = wp::team_lane(LW); i < m; i += LW)
            if (!(th < fth[i] || ph < fph[i])) ok = false;
        return tred_min(ok ? 1.0 : 0.0) > 0.5;
    }
    NMPC_PASS void filter_add(double th, double ph)
    {
        NMPC_LOCALS
        double *fth = wp::global_ptr(filter_base()), *fph = fth + NMPC_FILTER_CAP;
        if (l == 0) {
            const int slot = fn % NMPC_FILTER_CAP;
            fth[slot] = th; fph[slot] = ph;
            if (fn >= NMPC_FILTER_CAP) sm[SM_MISC + 2] += 1.0;
        }
        fn++;
        tsync();
    }
    static NMPC_DEV bool cmp_le(double lhs, double rhs, double bas) { return lhs - rhs <= 10.0 * 2.220446049250313e-16 * fabs(bas); }

    // ---------------------------------------------------------------------------------------
    // outputs in the reference layout, multipliers in CasADi's sign convention
    // ---------------------------------------------------------------------------------------
    NMPC_PASS void write_outputs(int st, int iter, double E0, double pinf, double dinf, double c0, double mu)
    {
        NMPC_LOCALS
        // g / lam_g layout: N + 1 blocks of [NS equality rows ; MQ inequality rows]; the obstacle scripts (family 1) have no inequality
        // rows in block 0 (first_scenario_mpc_obstacle_avoidance.py:109-125), so block k >= 1 starts at NS + (k - 1)(NS + MQ)
        const long long MQ = M + (long long)NR * nobs, n = (long long)NS * S + (long long)NC * N;
        const long long mg = family ? NS + (long long)N * (NS + MQ) : (long long)S * (NS + MQ);
        auto goff = [=](int b) -> long long { return family ? (b == 0 ? 0 : NS + (long long)(b - 1) * (NS + MQ)) : (long long)b * (NS + MQ); };
        double *x = P.x + inst * n;
        double *lx = P.lam_x ? P.lam_x + inst * n : nullptr;
        double *g = P.g ? P.g + inst * mg : nullptr;
        double *lg = P.lam_g ? P.lam_g + inst * mg : nullptr;
        double *zb = sm + SM_ZB, *cs = sm + SM_CS, *sn = sm + SM_SN;
        double fo = 0.0;
        for (int k = 0; k <= N; k++) {
            tsync();
            const bool zv = zvalid(k);
            double zk = zv ? row(R_Z, k)[l] : 0.0;
            zb[l] = zk;
            if (zv) {
                long long idx = isx ? (long long)k * NS + l : (long long)NS * S + (long long)k * NC + (l - NS);
                x[idx] = zk;
                if (lx) lx[idx] = (row(R_ZU, k)[l] - row(R_ZL, k)[l]) / df;
                if (k < N) { double e = zk - (TRK ? row(R_REF, k)[l] : xs_l); fo += 0.5 * qw * e * e; }
            }
            tsync();
            if (k < N && l < NR) { double s_, c_; wp::sincos_(zb[3 * l + 2], &s_, &c_); cs[l] = c_; sn[l] = s_; }
            tsync();
            if (isx) {
                if (k == 0) {
                    if (g) g[l] = zk - x0bar_l;
                    if (lg) lg[l] = row(R_YC, 0)[l] / df;
                }
                if (k < N) {
                    double v = zb[NS + 2 * rob];
                    double pred = comp == 0 ? zk + T * v * cs[rob] : (comp == 1 ? zk + T * v * sn[rob] : zk + T * zb[NS + 2 * rob + 1]);
                    if (g) g[goff(k + 1) + l] = row(R_Z, k + 1)[l] - pred;
                    if (lg) lg[goff(k + 1) + l] = row(R_YC, k + 1)[l] / df;
                }
            }
            if (isq) {
                if (k == 0 && !family) {
                    if (g) g[NS + l] = NMPC_DUMMY_ROW_VALUE;
                    if (lg) lg[NS + l] = row(R_YD, 0)[l] / df;
                }
                if (k < N) {
                    if (g) g[goff(k + 1) + NS + l] = rowg(zb, pi, pj, isobs, qob + k * qos).dv;
                    if (lg) lg[goff(k + 1) + NS + l] = row(R_YD, k + 1)[l] / df;
                }
            }
        }
        fo = tred_sum(fo);
        if (l == 0) {
            if (P.f) P.f[inst] = fo;
            if (P.status) P.status[inst] = st;
            if (P.iters) P.iters[inst] = iter;
            if (P.stats) {
                double *sp = P.stats + (long long)inst * NMPC_NSTATS;
                sp[NMPC_ST_KKT_ERR] = E0; sp[NMPC_ST_PRIMAL_INF] = pinf; sp[NMPC_ST_DUAL_INF] = dinf; sp[NMPC_ST_COMPL] = c0;
                sp[NMPC_ST_MU] = mu; sp[NMPC_ST_N_REG] = n_reg; sp[NMPC_ST_N_RESTO] = n_resto; sp[NMPC_ST_N_SOC] = n_soc;
                sp[NMPC_ST_N_FACTOR] = n_fact; sp[NMPC_ST_N_LS] = n_ls; sp[NMPC_ST_FILTER_EVICT] = sm[SM_MISC + 2];
            }
        }
        tsync();
    }

    // trial-point acceptance test shared by the line search and the second-order correction
    NMPC_DEV bool trial_ok(double th_t, double ph_t, double theta, double phi, double theta_max, double theta_min, double gbd,
                           double alpha_test, bool ftype) const
    {
        if (!(fin(th_t) && fin(ph_t)) || !cmp_le(th_t, theta_max, theta)) return false;
        bool ok;
        if (ftype && theta <= theta_min) ok = cmp_le(ph_t - phi, 1e-8 * alpha_test * gbd, phi);
        else ok = cmp_le(th_t, (1.0 - 1e-5) * theta, theta) || cmp_le(ph_t - phi, -1e-8 * theta, phi);
        return ok && filter_ok(th_t, ph_t);
    }

    // ---------------------------------------------------------------------------------------
    // Parametric sensitivity of a returned solution (nmpc_solution_vjp / nmpc_solution_jvp), centralized family only.  The
    // point (x, lam_x, lam_g) is loaded in place of an iterate, unscaled (df = 1, so the stored multipliers are CasADi's): the
    // bound multipliers split by sign into zL / zU, the slacks set to the row values at x, block 0's constant rows weighted 0.
    // factor<3> with mu = delta = 0 then builds K = [[W + Sx, J'], [J, -Ss^-1]] (W = Hessian of the Lagrangian, Sx / Ss the
    // interior-point weights |lam| / distance to the relaxed bound) and the forward pass solves K [dz; y] = -[g; c] for the
    // seeded g (R_GX) and c (R_CSOC; R_DSOC = 0: no row depends on p):
    //   reverse: g = -x_bar, c = 0                     ->  p_bar[x0bar] = y of block 0,  p_bar[ref] = 2Q / 2R times dz
    //   forward: g = d(grad f)/dp p_dot, c = dg/dp p_dot ->  x_dot = dz
    // A pivot <= 0 (wrong inertia: second-order sufficiency fails, the derivative is not defined) gives status 1 and NaN.
    // ---------------------------------------------------------------------------------------
    // the point (and, SEEDED, the seeds of sensitivity()) loaded in place of an iterate, then factor<3>; false when the bounds were
    // rejected (ok = false on entry) or a pivot is <= 0.  Unseeded, R_GX and R_CSOC are zero: K is the same, the right-hand side 0.
    template <bool SEEDED>
    NMPC_DEV bool sens_factor(const NmpcSensParams &SP, bool ok)
    {
        NMPC_LOCALS
        const long long n = (long long)NS * S + (long long)NC * N, blk = NS + M, np = TRK ? NS + (long long)N * NZ : 2 * NS;
        const double *x = SP.x + inst * n, *lx = SP.lam_x + inst * n, *lg = SP.lam_g + inst * (S * blk);
        const double *sd = SEEDED ? SP.seed + inst * (SP.reverse ? n : np) : nullptr;
        auto xidx = [=](int k) -> long long { return isx ? (long long)k * NS + l : (long long)NS * S + (long long)k * NC + (l - NS); };
        if (ok) {
            for (int k = 0; k <= N; k++) {
                const bool zv = zvalid(k);
                const double lam = zv ? lx[xidx(k)] : 0.0;
                row(R_Z, k)[l] = zv ? x[xidx(k)] : 0.0;
                row(R_ZL, k)[l] = (zv && brow(NMPC_BR_BL, k)[l] > -NMPC_INF) ? fmax(-lam, 0.0) : 0.0;
                row(R_ZU, k)[l] = (zv && brow(NMPC_BR_BU, k)[l] < NMPC_INF) ? fmax(lam, 0.0) : 0.0;
                row(R_YC, k)[l] = isx ? lg[k * blk + l] : 0.0;
                row(R_YD, k)[l] = isq ? lg[k * blk + NS + l] : 0.0;
                double g = 0.0;
                if (SEEDED) {
                    if (SP.reverse) g = zv ? -sd[xidx(k)] : 0.0;
                    else if (k < N && isz) g = -qw * (TRK ? sd[NS + k * NZ + l] : (isx ? sd[NS + l] : 0.0));
                }
                row(R_GX, k)[l] = g;
                row(R_CSOC, k)[l] = (SEEDED && !SP.reverse && k == 0 && isx) ? -sd[l] : 0.0;
                row(R_DSOC, k)[l] = 0.0;
            }
            tsync();
            for (int b = 0; b <= N; b++) {
                double s = NMPC_DUMMY_ROW_VALUE, vl = 0.0, vu = 0.0;
                if (isq && b > 0) {
                    const double yd = row(R_YD, b)[l];
                    s = rowg(row(R_Z, b - 1), pi, pj, false, nullptr).dv;
                    vl = brow(NMPC_BR_DL, b)[l] > -NMPC_INF ? fmax(-yd, 0.0) : 0.0;
                    vu = brow(NMPC_BR_DU, b)[l] < NMPC_INF ? fmax(yd, 0.0) : 0.0;
                }
                row(R_S, b)[l] = s; row(R_VL, b)[l] = vl; row(R_VU, b)[l] = vu;
            }
            tsync();
            trig_rows(row, l, N, 0.0, 0, false, R_TRIG);
            this->r_trig = R_TRIG; this->trig_valid = true;
            ok = factor<3>(0.0, 0.0, true);
        }
        return ok;
    }

    NMPC_PASS void sensitivity(const NmpcSensParams &SP)
    {
        NMPC_LOCALS
        static_assert(!OBS, "the obstacle families have no sensitivity pass");
        const long long n = (long long)NS * S + (long long)NC * N, np = TRK ? NS + (long long)N * NZ : 2 * NS;
        double *out = SP.out + inst * (SP.reverse ? np : n);
        auto xidx = [=](int k) -> long long { return isx ? (long long)k * NS + l : (long long)NS * S + (long long)k * NC + (l - NS); };
        const int berr = P.bound_err ? *P.bound_err : 0;
        const bool ok = sens_factor<true>(SP, berr == 0);
        if (ok) {
            StepInfo si;
            forward(0.0, 1.0, R_DZ, R_DS, R_YTC, R_YTD, si);
        }
        const double nan = (double)NAN;
        if (SP.reverse) {
            if (isx) out[l] = ok ? row(R_YTC, 0)[l] : nan;
            double acc = 0.0;
            for (int k = 0; k < N; k++) {
                const double a = ok ? row(R_DZ, k)[l] : nan;
                if (TRK && isz) out[NS + (long long)k * NZ + l] = qw * a;
                acc += a;
            }
            if (!TRK && isx) out[NS + l] = qw * acc;
        } else {
            for (int k = 0; k <= N; k++)
                if (zvalid(k)) out[xidx(k)] = ok ? row(R_DZ, k)[l] : nan;
        }
        if (SP.status && l == 0) SP.status[inst] = berr ? berr : (ok ? 0 : 1);
        tsync();
    }

    // ---------------------------------------------------------------------------------------
    // Jacobian of the solution with respect to the measured state x0bar = p[0:NS] (nmpc_solution_x0_jacobian): column j is
    // sensitivity()'s forward mode for p_dot = e_j.  That seed enters only through c of block 0 (R_CSOC row 0, which factor<3>
    // copies to R_RC row 0 after the sweep and nothing in the sweep reads): with zero seeds the factorisation, its feed-forward
    // terms and the block-0 rows are those of every column, so the point is factored once and each column is one forward pass
    // started from R_RC row 0 = -e_j.  Output SP.out: jac [B][NS][n], column j in x's layout (its X_0 rows are e_j); status and
    // NaN outputs as in sensitivity().
    // ---------------------------------------------------------------------------------------
    NMPC_PASS void sensitivity_x0(const NmpcSensParams &SP)
    {
        NMPC_LOCALS
        const long long n = (long long)NS * S + (long long)NC * N;
        double *jac = SP.out + inst * (NS * n);
        auto xidx = [=](int k) -> long long { return isx ? (long long)k * NS + l : (long long)NS * S + (long long)k * NC + (l - NS); };
        const int berr = P.bound_err ? *P.bound_err : 0;
        const bool ok = sens_factor<false>(SP, berr == 0);
        const double nan = (double)NAN;
        for (int j = 0; j < NS; j++) {
            if (ok) {
                if (isx) row(R_RC, 0)[l] = -(l == j ? 1.0 : 0.0);
                StepInfo si;
                forward(0.0, 1.0, R_DZ, R_DS, R_YTC, R_YTD, si);
            }
            double *out = jac + j * n;
            for (int k = 0; k <= N; k++)
                if (zvalid(k)) out[xidx(k)] = ok ? row(R_DZ, k)[l] : nan;
        }
        if (SP.status && l == 0) SP.status[inst] = berr ? berr : (ok ? 0 : 1);
        tsync();
    }

    // ---------------------------------------------------------------------------------------
    // hooks used by the shared interior-point driver (ipm_driver.cuh)
    // ---------------------------------------------------------------------------------------
    NMPC_DEV bool is_lead() const { return l == 0; }
    // Convoy mode (P.convoy > 0): the teams of a CTA meet at the start of every IPM iteration and
    // (P.convoy > 1) again before the forward pass, so that they run the same pass at about the same time and share its
    // instructions in the SM's instruction cache.  Every barrier also counts the working warps (an idle warp
    // contributes 0) -- see solve_kernel.
    NMPC_DEV void iter_sync() const { if (P.convoy) wp::cta_count(l == 0); }
    // (joining only PAIRS of warps at the second barrier was measured: 47.6 k against 50.7 k solves/s -- the aligned forward pass and
    // line search are worth more than the shorter wait)
    NMPC_DEV void mid_sync() const { if (P.convoy > 1) wp::cta_count(l == 0); }
    NMPC_DEV bool factor_m(int mode, double mu, double delta, bool soc)
    {
        return mode == 0 ? factor<0>(mu, delta, soc) : (mode == 1 ? factor<1>(mu, delta, soc) : factor<2>(mu, delta, soc));
    }
    NMPC_DEV void eval(bool full, double mu, double alpha, int rdz, int rds, bool trial, bool socacc, double asoc, EvalOut &E)
    {
        eval_pass_rt(full, mu, alpha, rdz, rds, trial, socacc, asoc, E);
    }
    // largest |y| over the equality and inequality multipliers (least-squares initialisation)
    NMPC_DEV double mult_absmax()
    {
        double ymax = 0.0;
        for (int k = 0; k <= N; k++) ymax = fmax(ymax, fmax(isx ? fabs(row(R_YC, k)[l]) : 0.0, (isq) ? fabs(row(R_YD, k)[l]) : 0.0));
        return tred_max(ymax);
    }
    NMPC_DEV void mult_zero()
    {
        for (int k = 0; k <= N; k++) { row(R_YC, k)[l] = 0.0; row(R_YD, k)[l] = 0.0; }
    }
    NMPC_DEV bool bounds_rejected()
    {
        if (P.bound_err && *P.bound_err) {  // bounds rejected by prep_bounds_kernel: report, do not solve
            if (l == 0) { if (P.status) P.status[inst] = *P.bound_err; if (P.iters) P.iters[inst] = 0; }
            return true;
        }
        return false;
    }
    NMPC_DEV void run() { ipm_run(*this); }
};
