// CTA-per-instance dense-block solver for large swarms (Nr > 10, e.g. the 64-robot configuration).
//
// Same NLP and the same interior-point iteration (ipm_driver.cuh) as the warp-per-instance solver, for the case where
// a stage of the KKT system no longer fits the lanes of a warp: the stage blocks become dense matrices
// (64 robots: P 192 x 192, control block 128 x 128, 2016 pair rows per stage).  Replaces, for one instance,
//     sol = solver(x0=, p=, lbx=, ubx=, lbg=, ubg=)          centralized_six_robots_implementation.py:432
// built by the many-robot scripts (mpc_online_casadi_tb3_ten_robots...py:169-380 is the largest in the reference).
//
// Mapping: one CTA (BLOCK_THREADS threads) per instance, instances pulled from an atomic queue.  Vectors live in a
// per-CTA scratch area in global memory (L2 resident) as [row][stage][W] with W >= max(5 Nr, M); the vector passes are
// flat thread-strided loops over (stage, variable / pair).  The Riccati factorisation keeps the control block of the
// stage matrix in shared memory:
//     M = H~ + [A B]' P+ [A B]     assembled per robot pair from the 3x3 blocks of P+ (A, B are unicycle-sparse)
//     M_uu = L L'                  blocked right-looking Cholesky in place in shared memory, 32-column panels: the diagonal block by
//                                  one warp in registers, the rows below by substitution, the trailing update as 8 x 8 tiles on the
//                                  FP64 tensor instruction; a pivot <= 0 is IPOPT's wrong-inertia signal
//     Y = L^-1 [M_ux | m_u]        Y resident in shared memory; with the inverses of the 32 x 32 diagonal blocks, V = blockdiag(Linv) B
//                                  and W_IJ = Linv_II L_IJ, the block rows are Y_I = V_I - sum_{J < I} W_IJ Y_J (tensor instruction)
//     P = M_xx - Y'Y, p = m_x - Y' y_m     upper 8 x 8 tiles of the Gram matrix of [Y | y_m] (tensor instruction), mirrored
// and the forward pass applies  du = -L^-T (Y dx + y_m)  with L staged into shared memory by a bulk copy.  FP64 has no tcgen05 kind; the
// legacy DMMA (mma.sync m8n8k4 f64) shares the DFMA pipe and its peak on B200 (tools/probe_fp64_mix.cu), so it does not raise the
// roofline -- it is used because its fragments need a quarter of the shared-memory traffic of 4 x 4 register tiles.
#pragma once
#include "nmpc_internal.h"
#include "ipm_driver.cuh"
#include "solver_body.cuh"

#define NMPC_BLOCK_THREADS 512
// cycle counters of CTA 0 (thread 0) per phase of the dense-block solver; read with nmpc_debug_block_profile()
__device__ long long g_block_prof[16];
#define NMPC_PROF_BEGIN long long prof_t0_ = clock64();
#define NMPC_PROF(slot) do { if (blockIdx.x == 0 && threadIdx.x == 0) { long long t_ = clock64(); g_block_prof[slot] += t_ - prof_t0_; prof_t0_ = t_; } } while (0)
#define NMPC_BPASS __device__ __noinline__

// Inside a pass the solver object lives in local memory and its pointers are generic: shadow them with locals that carry
// their address space (shared / global), so that the compiler emits LDS / LDG instead of generic loads.
#define NMPC_BLK_LOCALS                                                                                                \
    double *const sm = wp::shared_ptr(this->sm);                                                                       \
    double *const ws = wp::global_ptr(this->ws);                                                                       \
    const double *const BL = wp::global_ptr(this->BL), *const BU = wp::global_ptr(this->BU),                            \
                 *const CE = wp::global_ptr(this->CE), *const DL = wp::global_ptr(this->DL),                            \
                 *const DU = wp::global_ptr(this->DU), *const pp = wp::global_ptr(this->pp);                            \
    const int *const pairs = wp::global_ptr(this->pairs);                                                              \
    const double *const obs = wp::global_ptr(this->obs);                                                               \
    const int Mp = this->Mp, nobs = this->nobs, ostr = this->ostr;                                                     \
    double *const Pall = wp::global_ptr(this->Pall), *const Yall = wp::global_ptr(this->Yall),                          \
                 *const Lall = wp::global_ptr(this->Lall),                                                             \
                 *const Wg = wp::global_ptr(this->Wg);                                                                 \
    const int S = this->S, W = this->W, N = this->N, Nr = this->Nr, ns = this->ns, nc = this->nc, nz = this->nz,        \
              M = this->M, tid = this->tid, nt = this->nt;                                                             \
    auto row = [=](int r, int k) -> double * { return ws + ((long long)r * S + k) * W; };                              \
    (void)sm; (void)ws; (void)BL; (void)BU; (void)CE; (void)DL; (void)DU; (void)pp; (void)pairs; (void)Pall;            \
    (void)Yall; (void)Lall; (void)Wg; (void)S; (void)W; (void)N; (void)Nr; (void)ns; (void)nc; (void)nz; (void)M;       \
    (void)tid; (void)nt; (void)row; (void)obs; (void)Mp; (void)nobs; (void)ostr;

struct BlockSolver {
    enum Row {
        R_Z, R_ZL, R_ZU, R_DZ, R_DZ2, R_GX, R_YC, R_YTC, R_YTC2, R_RC, R_CSOC, R_COEF, R_COEF2, R_LIN, R_DGV,
        R_S, R_VL, R_VU, R_YD, R_DS, R_DS2, R_YTD, R_YTD2, R_DSOC, R_GXQ, R_GYQ, R_RD, R_DQ, R_GS,
        R_PXX, R_PYY, R_PXY, R_PHX, R_PHY, R_TRIG, R_TRIG2, R_ZT, R_ST,
        R_COUNT
    };
    struct EvalOut { double pinf, viol, dinf, c0, cmu, ysum, zsum, theta, f, slog, sdamp; };
    struct StepInfo { double ap, az, gbd, tiny; };
    typedef WarpSolver<1> WS;   // scalar helpers (push_in, slack_step_terms, cmp_le, fin) are shared with the warp solver

    const NmpcSolveParams &P;
    double *sm, *ws;
    int Nr, N, S, ns, nc, nz, M, W, tid, nt, inst, fn;   // M: inequality rows per block = pair rows + obstacle rows
    int Mp, nobs, family;                                 // pair rows, obstacles per robot, row layout (0 centralized, 1 obstacles)
    const double *obs;                                    // [nobs][3] of stage 0: centre x, y, clearance radius
    int ostr;                                             // doubles from one stage's obstacle table to the next (0: static obstacles)
    int nref, rstr;                                       // reference in p after x0bar: variables per stage, stride (see ref())
    const double *BL, *BU, *CE, *DL, *DU, *pp;
    const int *pairs;
    double *Pall, *Yall, *Lall, *Wg;   // Wg: Linv_II L_IJ blocks of the stage being factored (see factor, step D)
    int ncp;   // nc rounded up to a multiple of 32 (blocked triangular solves)
    int ldy;   // leading dimension of Y_k and of [M_ux | m_u]: the smallest value >= ns + 1 that is 4 mod 8 (conflict-free DMMA fragment loads)
    double T, df, ny_nzb, nzb_cnt;
    int n_reg, n_resto, n_soc, n_fact, n_ls;
    // shared-memory carve-up (doubles)
    static constexpr int SM_MBAR = 32 * 12 + 16 + 16 + 4;   // = SM_MISC + 4: the CTA's mbarrier (initialised once per kernel)
    unsigned bar_phase = 0;
    int SM_RED, SM_FTH, SM_FPH, SM_MISC, SM_DZB, SM_DXN, SM_TB, SM_XB, SM_DINV, SM_PR, SM_CS, SM_DS, SM_MUU;

    static NMPC_HD int row_width(int Nr, int nobs = 0) { int nz = 5 * Nr, M = Nr * (Nr - 1) / 2 + Nr * nobs, w = nz > M ? nz : M; return (w + 31) & ~31; }
    static NMPC_HD long long ws_doubles(int Nr, int N, int nobs = 0)
    {
        const long long S = N + 1, ns = 3 * Nr, nc = 2 * Nr, W = row_width(Nr, nobs);
        const long long ldy = ((ns + 4) & ~7LL) + 4;
        const long long ncp = (nc + 31) & ~31LL;
        return (long long)R_COUNT * S * W + ((S * ns * ns + 1) & ~1LL) + (long long)N * nc * ldy + (long long)N * ncp * ncp   // every block 16-byte aligned
               + (ncp / 32) * (ncp / 32 - 1) / 2 * 1024 + 2 * NMPC_FILTER_CAP;   // the filter (theta values, then phi values), see filter_add
    }
    static NMPC_HD long long sm_doubles(int Nr)
    {
        const long long ns = 3 * Nr, nc = 2 * Nr, nz = 5 * Nr, ncp = (nc + 31) & ~31LL, ns4 = (ns + 3) & ~3LL;
        const long long a = ncp * (ncp + 4), b = ((nc + 3) & ~3LL) * (((ns + 4) & ~7LL) + 4);   // Cholesky factor (leading dimension ncp + 1: conflict-free columns), then Y resident for the triangular solve and the rank-k update
        (void)ns4;
        return 32 * 12 + 16 + 16 + 8 + nz + ns + 3 * ncp + ns + 7 * Nr + (a > b ? a : b) + 16;
    }

    __device__ BlockSolver(const NmpcSolveParams &p, double *smem, double *wsp) : P(p), sm(smem), ws(wsp) {}

    static __device__ __forceinline__ void tsync() { __syncthreads(); }
    __device__ __forceinline__ double *row(int r, int k) const { return ws + ((long long)r * S + k) * W; }
    __device__ __forceinline__ bool is_lead() const { return tid == 0; }
    __device__ __forceinline__ void iter_sync() const {}
    __device__ __forceinline__ void mid_sync() const {}
    __device__ __forceinline__ int pairidx(int a, int b) const { return a * (2 * Nr - a - 1) / 2 + (b - a - 1); }
    __device__ __forceinline__ double qw(int l) const { return l < ns ? 2.0 * P.Q[l % 3] : 2.0 * P.R[(l - ns) & 1]; }
    // reference of variable l at stage k: the setpoint xs (nref = ns, rstr = 0), or Z[k] of a tracking handle (nref = rstr = nz)
    __device__ __forceinline__ double ref(int k, int l) const { return l < nref ? pp[ns + k * rstr + l] : 0.0; }
    __device__ __forceinline__ double gradf(int k, int l, double z) const { return k < N ? qw(l) * (z - ref(k, l)) : 0.0; }
    __device__ __forceinline__ int nvalid(int k) const { return k < N ? nz : ns; }

    // FP64 tensor instruction: D (8 x 8) += A (8 x 4) B (4 x 8) over a warp.  Lane l = 4 g + t holds A[g][t], B[t][g] and D[g][2 t], D[g][2 t + 1].
    // On B200 it has the DFMA pipe's peak (nmpc_probe_dmma) but needs a quarter of the operand traffic of 4 x 4 register tiles.
    static __device__ __forceinline__ void dmma(double (&c)[2], double a, double b)
    {
        asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
    }

    // block-wide reduction of K values at once; bit i of maxmask: max (else sum); bit i of minmask: min
    template <int K>
    __device__ void breduce(double (&v)[K], unsigned maxmask)
    {
        NMPC_BLK_LOCALS
        double *red = sm + SM_RED;
        const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
#pragma unroll
        for (int i = 0; i < K; i++) {
            double x = v[i];
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) {
                double y = __shfl_xor_sync(0xffffffffu, x, m);
                x = (maxmask >> i & 1u) ? fmax(x, y) : x + y;
            }
            v[i] = x;
        }
        __syncthreads();
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < K; i++) red[wid * 12 + i] = v[i];
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < K; i++) {
            double x = red[i];
            for (int w = 1; w < nw; w++) { double y = red[w * 12 + i]; x = (maxmask >> i & 1u) ? fmax(x, y) : x + y; }
            v[i] = x;
        }
        __syncthreads();
    }
    __device__ double bsum(double x) { double v[1] = {x}; breduce<1>(v, 0u); return v[0]; }
    __device__ double bmax(double x) { double v[1] = {x}; breduce<1>(v, 1u); return v[0]; }

    // ---------------------------------------------------------------------------------------
    __device__ void setup(int instance)
    {
        inst = instance; Nr = P.Nr; N = P.N; S = N + 1; ns = 3 * Nr; nc = 2 * Nr; nz = 5 * Nr;
        Mp = Nr * (Nr - 1) / 2; nobs = P.nobs; family = P.family; M = Mp + Nr * nobs;
        W = row_width(Nr, nobs); T = P.T; tid = threadIdx.x; nt = blockDim.x;
        const double *br = P.brows + (long long)inst * P.bstride;
        BL = br + (long long)NMPC_BR_BL * S * W; BU = br + (long long)NMPC_BR_BU * S * W;
        CE = br + (long long)NMPC_BR_CE * S * W; DL = br + (long long)NMPC_BR_DL * S * W;
        DU = br + (long long)NMPC_BR_DU * S * W;
        pp = P.p + (long long)inst * P.np;
        // Reference after x0bar: one setpoint xs, or Z[N][nz] of a tracking handle; then, with the obstacles in p, one [nobs][3]
        // table per stage.  The four layouts and their np:
        //     [x0bar; xs]                 2 ns                 [x0bar; Z]         ns + N nz
        //     [x0bar; xs; O[N]]           2 ns + 3 N nobs      [x0bar; Z; O[N]]   ns + N nz + 3 N nobs
        // Since N nz = 5 Nr N never equals ns = 3 Nr, a tracking np never equals the setpoint np with the same obstacle block.
        // (Told apart by np rather than by a flag in NmpcSolveParams: a larger parameter block would change the frame, and so
        // the code, of every warp-path kernel, which copies it to local memory.)
        const bool trk = P.np == ns + N * nz + (P.obs_in_p ? 3 * N * nobs : 0);
        nref = trk ? nz : ns; rstr = trk ? nz : 0;
        // obstacles in p: after x0bar and the reference, one table per stage; else the handle's table at every stage
        obs = P.obs_in_p ? pp + ns + (trk ? N * nz : ns) : P.obs; ostr = P.obs_in_p ? 3 * nobs : 0;
        pairs = P.pairs;
        Pall = ws + (long long)R_COUNT * S * W;
        ldy = ((ns + 4) & ~7) + 4; ncp = (nc + 31) & ~31;
        Yall = Pall + (((long long)S * ns * ns + 1) & ~1LL);
        Lall = Yall + (long long)N * nc * ldy;
        Wg = Lall + (long long)N * ncp * ncp;
        SM_RED = 0; SM_FTH = 32 * 12; SM_FPH = SM_FTH + 16; SM_MISC = SM_FPH + 16; SM_DZB = SM_MISC + 8; SM_DXN = SM_DZB + nz;
        SM_TB = SM_DXN + ns; SM_XB = SM_TB + ncp; SM_DINV = SM_XB + ncp; SM_PR = SM_DINV + ncp; SM_CS = SM_PR + ns; SM_DS = SM_CS + 2 * Nr; SM_MUU = (SM_DS + 5 * Nr + 1) & ~1;
        df = 1.0; fn = 0;
        n_reg = n_resto = n_soc = n_fact = n_ls = 0;
        if (tid == 0) sm[SM_MISC + 2] = 0.0;   // filter evictions
        __syncthreads();
    }
    __device__ bool bounds_rejected()
    {
        if (P.bound_err && *P.bound_err) {
            if (tid == 0) { if (P.status) P.status[inst] = *P.bound_err; if (P.iters) P.iters[inst] = 0; }
            return true;
        }
        return false;
    }

    // cos / sin of every heading of the evaluation point: row(rt,k)[i] = cos, row(rt,k)[Nr+i] = sin
    __device__ void trig_rows(double alpha, int rdz, bool trial, int rt)
    {
        NMPC_BLK_LOCALS
        for (int idx = tid; idx < N * Nr; idx += nt) {
            const int k = idx / Nr, i = idx - k * Nr;
            double th = row(R_Z, k)[3 * i + 2];
            if (trial) th += alpha * row(rdz, k)[3 * i + 2];
            double s_, c_;
            sincos(th, &s_, &c_);
            row(rt, k)[i] = c_; row(rt, k)[Nr + i] = s_;
        }
        __syncthreads();
    }

    // starting point: objective scaling, push into bounds, slacks, bound multipliers (IPOPT defaults)
    NMPC_BPASS void init_point()
    {
        NMPC_BLK_LOCALS
        const long long n = (long long)ns * S + (long long)nc * N;
        const double *x0 = P.x0 + inst * n;
        const nmpc_opts &o = P.o;
        double gmax = 0.0;
        for (int idx = tid; idx < S * nz; idx += nt) {
            const int k = idx / nz, l = idx - k * nz;
            const double z = l < ns ? x0[k * ns + l] : (k < N ? x0[ns * S + k * nc + (l - ns)] : 0.0);
            gmax = fmax(gmax, fabs(gradf(k, l, z)));
            row(R_Z, k)[l] = z;
        }
        gmax = bmax(gmax);
        df = gmax > o.nlp_scaling_max_gradient ? fmax(o.nlp_scaling_max_gradient / gmax, 1e-8) : 1.0;
        double cnt_z = 0.0, cnt_y = tid == 0 ? (double)(ns * S) : 0.0;
        for (int idx = tid; idx < S * W; idx += nt) {
            const int k = idx / W, l = idx - k * W;
            if (l < nz) {
                const double lo = BL[k * W + l], hi = BU[k * W + l];
                row(R_Z, k)[l] = WS::push_in(row(R_Z, k)[l], lo, hi, o.bound_push, o.bound_frac);
                const bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
                row(R_ZL, k)[l] = hl ? o.bound_mult_init_val : 0.0;
                row(R_ZU, k)[l] = hu ? o.bound_mult_init_val : 0.0;
                cnt_z += (hl ? 1.0 : 0.0) + (hu ? 1.0 : 0.0);
            }
            row(R_YC, k)[l] = 0.0; row(R_YD, k)[l] = 0.0; row(R_CSOC, k)[l] = 0.0; row(R_DSOC, k)[l] = 0.0;
        }
        __syncthreads();
        for (int idx = tid; idx < S * M; idx += nt) {
            const int b = idx / M, q = idx - b * M;
            const double lo = DL[b * W + q], hi = DU[b * W + q];
            const bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
            double dv = NMPC_DUMMY_ROW_VALUE;
            if (b > 0) dv = rowgeom(row(R_Z, b - 1), q, Mp, nobs, pairs, obs + (b - 1) * ostr).dv;
            row(R_S, b)[q] = (hl || hu) ? WS::push_in(dv, lo, hi, o.bound_push, o.bound_frac) : dv;
            row(R_VL, b)[q] = hl ? o.bound_mult_init_val : 0.0;
            row(R_VU, b)[q] = hu ? o.bound_mult_init_val : 0.0;
            cnt_z += (hl ? 1.0 : 0.0) + (hu ? 1.0 : 0.0);
            cnt_y += (hl || hu) ? 1.0 : 0.0;
        }
        double v[2] = {cnt_z, cnt_y};
        breduce<2>(v, 0u);
        nzb_cnt = v[0]; ny_nzb = v[1] + v[0];
        trig_rows(0.0, 0, false, R_TRIG);
    }

    // one predicted state component: X_k + T f(X_k, U_k), component l of the state vector
    __device__ __forceinline__ double predict(const double *zr, const double *tr, int l) const
    {
        const int rob = l / 3, comp = l - 3 * rob;
        const double v = zr[ns + 2 * rob];
        return comp == 0 ? zr[l] + T * v * tr[rob] : (comp == 1 ? zr[l] + T * v * tr[Nr + rob] : zr[l] + T * zr[ns + 2 * rob + 1]);
    }

    // Inequality row q of a block evaluated on the stage vector zr.  Rows q < Mp are the pairwise squared distances
    // (centralized_six_robots_implementation.py:288-306); rows q >= Mp are the static circular obstacles of family F,
    // sqrt((x - ox)^2 + (y - oy)^2) - r_rob - r_obs (first_scenario_mpc_obstacle_avoidance.py:125), nobs per robot;
    // obs: the obstacle table [nobs][3] of the stage zr belongs to.
    // i, j: robots (j = -1 for an obstacle row); (gx, gy): gradient w.r.t. (x_i, y_i) (negated for robot j);
    // (hxx, hyy, hxy): second derivatives w.r.t. (x_i, y_i).
    struct RowG { double dv, gx, gy, hxx, hyy, hxy; int i, j; };
    static __device__ __forceinline__ RowG rowgeom(const double *zr, int q, int Mp, int nobs, const int *pairs, const double *obs)
    {
        RowG r;
        if (q < Mp) {
            r.i = pairs[2 * q]; r.j = pairs[2 * q + 1];
            const double dx = zr[3 * r.i] - zr[3 * r.j], dy = zr[3 * r.i + 1] - zr[3 * r.j + 1];
            r.dv = dx * dx + dy * dy; r.gx = 2.0 * dx; r.gy = 2.0 * dy; r.hxx = 2.0; r.hyy = 2.0; r.hxy = 0.0;
        } else {
            const int e = q - Mp, o = e % nobs;
            r.i = e / nobs; r.j = -1;
            const double dx = zr[3 * r.i] - obs[3 * o], dy = zr[3 * r.i + 1] - obs[3 * o + 1];
            const double rho = sqrt(dx * dx + dy * dy), ir = 1.0 / rho;
            r.gx = dx * ir; r.gy = dy * ir; r.dv = rho - obs[3 * o + 2];
            r.hxx = (1.0 - r.gx * r.gx) * ir; r.hyy = (1.0 - r.gy * r.gy) * ir; r.hxy = -r.gx * r.gy * ir;
        }
        return r;
    }
    // offset of block k in the flat g / lam_g vectors: family 1 has no inequality rows in block 0
    __device__ __forceinline__ long long goff(int k) const { return family ? (k == 0 ? 0 : ns + (long long)(k - 1) * (ns + M)) : (long long)k * (ns + M); }

    // ---------------------------------------------------------------------------------------
    // residuals / merit quantities at the iterate (full) or at a trial point z + alpha dz
    // ---------------------------------------------------------------------------------------
    NMPC_BPASS void eval(bool full, double mu, double alpha, int rdz, int rds, bool trial, bool socacc, double asoc, EvalOut &E)
    {
        NMPC_BLK_LOCALS
        const double kd = P.o.kappa_d;
        NMPC_PROF_BEGIN
        const int rt = trial ? R_TRIG2 : R_TRIG, rz = trial ? R_ZT : R_Z, rs = trial ? R_ST : R_S;
        if (trial) {   // materialise the trial point once
            for (int idx = tid; idx < S * W; idx += nt) {
                const int k = idx / W, l = idx - k * W;
                if (l < nz) row(R_ZT, k)[l] = l < nvalid(k) ? row(R_Z, k)[l] + alpha * row(rdz, k)[l] : 0.0;
                if (l < M) row(R_ST, k)[l] = row(R_S, k)[l] + alpha * row(rds, k)[l];
            }
        }
        trig_rows(alpha, rdz, trial, rt);   // ends with a barrier
        double pinf = 0, viol = 0, dinf = 0, c0 = 0, cmu = 0, ysum = 0, zsum = 0, th = 0, fo = 0, sdamp = 0, slog = 0;
        // ---- equality rows ----
        for (int idx = tid; idx < S * ns; idx += nt) {
            const int k = idx / ns, l = idx - k * ns;
            double c;
            if (k == 0) c = row(rz, 0)[l] - pp[l] - CE[l];
            else c = row(rz, k)[l] - predict(row(rz, k - 1), row(rt, k - 1), l) - CE[k * W + l];
            pinf = fmax(pinf, fabs(c)); th += fabs(c); viol = fmax(viol, fabs(c));
            if (socacc) row(R_CSOC, k)[l] = asoc * row(R_CSOC, k)[l] + c;
            if (full) ysum += fabs(row(R_YC, k)[l]);
        }
        // ---- inequality rows ----
        for (int idx = tid; idx < S * M; idx += nt) {
            const int b = idx / M, q = idx - b * M;
            // every load of the row is issued before the first branch on its bounds: behind the branch they are a second dependent
            // L2 / DRAM round trip per row (the compiler may not speculate them)
            const double lo = DL[b * W + q], hi = DU[b * W + q];
            const double s = row(rs, b)[q];
            const double yd_ = full ? row(R_YD, b)[q] : 0.0, vl_ = full ? row(R_VL, b)[q] : 0.0, vu_ = full ? row(R_VU, b)[q] : 0.0;
            const double dsoc_ = socacc ? row(R_DSOC, b)[q] : 0.0;
            double dv = NMPC_DUMMY_ROW_VALUE;
            if (b > 0) dv = rowgeom(row(rz, b - 1), q, Mp, nobs, pairs, obs + (b - 1) * ostr).dv;
            const bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
            if (!(hl || hu)) continue;
            const double dms = dv - s;
            pinf = fmax(pinf, fabs(dms)); th += fabs(dms);
            viol = fmax(viol, fmax(lo - dv, dv - hi));
            if (socacc) row(R_DSOC, b)[q] = asoc * dsoc_ + dms;
            if (hl) slog += log(s - lo);
            if (hu) slog += log(hi - s);
            if (hl && !hu) sdamp += s - lo;
            if (hu && !hl) sdamp += hi - s;
            if (full) {
                const double yd = yd_, vl = vl_, vu = vu_;
                ysum += fabs(yd);
                double t = -yd - vl + vu;
                if (hl && !hu) t += kd * mu;
                if (hu && !hl) t -= kd * mu;
                dinf = fmax(dinf, fabs(t));
                if (hl) { double u = (s - lo) * vl; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(vl); }
                if (hu) { double u = (hi - s) * vu; c0 = fmax(c0, fabs(u)); cmu = fmax(cmu, fabs(u - mu)); zsum += fabs(vu); }
            }
        }
        // ---- variable bounds, objective, stationarity ----
        for (int idx = tid; idx < S * nz; idx += nt) {
            const int k = idx / nz, l = idx - k * nz;
            if (l >= nvalid(k)) continue;
            const double *zr = row(rz, k);
            const double zk = zr[l], lo = BL[k * W + l], hi = BU[k * W + l];
            const bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
            if (hl) slog += log(zk - lo);
            if (hu) slog += log(hi - zk);
            if (hl && !hu) sdamp += zk - lo;
            if (hu && !hl) sdamp += hi - zk;
            if (k < N) { const double e = zk - ref(k, l); fo += 0.5 * qw(l) * e * e; }
            if (full) {
                const double zl = row(R_ZL, k)[l], zu = row(R_ZU, k)[l];
                double r = df * gradf(k, l, zk) - zl + zu;
                if (hl && !hu) r += kd * mu;
                if (hu && !hl) r -= kd * mu;
                const bool isx = l < ns;
                const int rob = isx ? l / 3 : (l - ns) / 2, comp = isx ? l - 3 * rob : (l - ns) & 1;
                if (isx) r += row(R_YC, k)[l];
                if (k < N) {
                    const double *ycn = row(R_YC, k + 1), *tr = row(rt, k);
                    const double csr = tr[rob], snr = tr[Nr + rob];
                    if (isx) {
                        if (comp == 2) {
                            const double v = zr[ns + 2 * rob];
                            r -= ycn[l] + (-T * v * snr) * ycn[3 * rob] + (T * v * csr) * ycn[3 * rob + 1];
                        } else {
                            r -= ycn[l];
                            const double *ydn = row(R_YD, k + 1);
                            for (int j = 0; j < Nr; j++) {
                                if (j == rob) continue;
                                const int q = rob < j ? pairidx(rob, j) : pairidx(j, rob);
                                r += 2.0 * (zk - zr[3 * j + comp]) * ydn[q];
                            }
                            for (int o = 0; o < nobs; o++) {   // static obstacles of this robot
                                const int q = Mp + rob * nobs + o;
                                const RowG rg = rowgeom(zr, q, Mp, nobs, pairs, obs + k * ostr);
                                r += (comp == 0 ? rg.gx : rg.gy) * ydn[q];
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
        NMPC_PROF(7);
        double v[11] = {pinf, viol, dinf, c0, cmu, ysum, zsum, th, fo, slog, sdamp};
        breduce<11>(v, 0x1Fu);   // first five are maxima
        E.pinf = v[0]; E.viol = v[1]; E.theta = v[7]; E.f = v[8]; E.slog = v[9]; E.sdamp = v[10];
        if (full) { E.dinf = v[2]; E.c0 = v[3]; E.cmu = v[4]; E.ysum = v[5]; E.zsum = v[6]; }
    }

    // barrier Hessian / gradient pieces of one variable or slack (mode 0: primal-dual, 1: least squares, 2: restoration)
    static __device__ __forceinline__ void sig_g(int mode, double kd, double v, double lo, double hi, double ml, double mu_, double mu,
                                                 double g0, double &sig, double &g)
    {
        const bool hl = lo > -NMPC_INF, hu = hi < NMPC_INF;
        if (mode == 1) { sig = 1.0; g = g0 - ml + mu_; return; }
        sig = 0.0; g = mode == 0 ? g0 : 0.0;
        if (hl) { const double r = 1.0 / (v - lo); sig += mode == 0 ? ml * r : mu * r * r; g -= mu * r; }
        if (hu) { const double r = 1.0 / (hi - v); sig += mode == 0 ? mu_ * r : mu * r * r; g += mu * r; }
        if (mode == 0) {
            if (hl && !hu) g += kd * mu;
            if (hu && !hl) g -= kd * mu;
        }
    }

    // ---------------------------------------------------------------------------------------
    // K3: backward Riccati sweep with dense stage blocks.  false = wrong inertia (a control pivot <= 0).
    // ---------------------------------------------------------------------------------------
    __device__ bool factor_m(int mode, double mu, double delta, bool soc)
    {
        return factor(mode, mu, delta, soc);
    }
    NMPC_BPASS bool factor(int mode, double mu, double delta, bool soc)
    {
        NMPC_BLK_LOCALS
        const double zeta = mode == 2 ? sqrt(mu) : 0.0, kd = P.o.kappa_d;
        double *Muu = sm + SM_MUU, *prv = sm + SM_PR, *colb = sm + SM_TB, *dinv = sm + SM_DINV;   // colb: 2 ncp doubles (SM_TB, SM_XB contiguous)
        n_fact++;
        __syncthreads();
        NMPC_PROF_BEGIN
        // ---- stage-parallel part: barrier terms, coefficients, residuals, condensed inequality blocks ----
        for (int idx = tid; idx < S * nz; idx += nt) {
            const int k = idx / nz, l = idx - k * nz;
            double sig = 0.0, gx = 0.0, dg = 0.0;
            if (l < nvalid(k)) {
                const double zk = row(R_Z, k)[l];
                sig_g(mode, kd, zk, BL[k * W + l], BU[k * W + l], row(R_ZL, k)[l], row(R_ZU, k)[l], mu, df * gradf(k, l, zk), sig, gx);
                dg = sig + delta + zeta;
                if (mode == 0 && k < N) dg += df * qw(l);
            }
            row(R_GX, k)[l] = gx; row(R_DGV, k)[l] = dg;
        }
        for (int idx = tid; idx < N * Nr; idx += nt) {
            const int k = idx / Nr, i = idx - k * Nr;
            const double v = row(R_Z, k)[ns + 2 * i], c_ = row(R_TRIG, k)[i], s_ = row(R_TRIG, k)[Nr + i];
            double *cf = row(R_COEF, k), *cf2 = row(R_COEF2, k);
            cf[i] = -T * v * s_; cf[Nr + i] = T * v * c_; cf[2 * Nr + i] = T * c_; cf[3 * Nr + i] = T * s_;
            if (mode == 0) {
                const double lx = row(R_YC, k + 1)[3 * i], ly = row(R_YC, k + 1)[3 * i + 1];
                cf2[i] = T * (lx * s_ - ly * c_); cf2[Nr + i] = T * v * (lx * c_ + ly * s_);
            } else { cf2[i] = 0.0; cf2[Nr + i] = 0.0; }
        }
        for (int idx = tid; idx < S * ns; idx += nt) {
            const int k = idx / ns, l = idx - k * ns;
            double rc = 0.0;
            if (mode != 1) {
                if (soc) rc = row(R_CSOC, k)[l];
                else if (k == 0) rc = row(R_Z, 0)[l] - pp[l] - CE[l];
                else rc = row(R_Z, k)[l] - predict(row(R_Z, k - 1), row(R_TRIG, k - 1), l) - CE[k * W + l];
            }
            row(R_RC, k)[l] = rc;
        }
        for (int idx = tid; idx < S * M; idx += nt) {
            const int b = idx / M, q = idx - b * M;
            double pxx = 0, pyy = 0, pxy = 0, phx = 0, phy = 0, gxq = 0, gyq = 0, rd = 0, Dq = 0, gs = 0;
            // (all loads of the row before the branch on its bounds, see eval)
            const double lo = DL[b * W + q], hi = DU[b * W + q];
            const double s = row(R_S, b)[q], vl_ = row(R_VL, b)[q], vu_ = row(R_VU, b)[q];
            const double dsoc_ = (soc && mode != 1) ? row(R_DSOC, b)[q] : 0.0, yd_ = mode == 0 ? row(R_YD, b)[q] : 0.0;
            RowG rg;
            rg.gx = rg.gy = rg.hxx = rg.hyy = rg.hxy = 0.0; rg.dv = NMPC_DUMMY_ROW_VALUE;
            if (b > 0) rg = rowgeom(row(R_Z, b - 1), q, Mp, nobs, pairs, obs + (b - 1) * ostr);
            if (lo > -NMPC_INF || hi < NMPC_INF) {
                const double dv = rg.dv, hxx = rg.hxx, hyy = rg.hyy, hxy = rg.hxy;
                gxq = rg.gx; gyq = rg.gy;
                double sigs;
                sig_g(mode, kd, s, lo, hi, vl_, vu_, mu, 0.0, sigs, gs);
                rd = mode == 1 ? 0.0 : (soc ? dsoc_ : dv - s);
                Dq = sigs + delta;
                const double hq = Dq * rd + gs, yq = yd_;   // multiplier times the row's own curvature
                pxx = Dq * gxq * gxq + yq * hxx; pyy = Dq * gyq * gyq + yq * hyy; pxy = Dq * gxq * gyq + yq * hxy;
                phx = gxq * hq; phy = gyq * hq;
            }
            row(R_GXQ, b)[q] = gxq; row(R_GYQ, b)[q] = gyq; row(R_RD, b)[q] = rd; row(R_DQ, b)[q] = Dq; row(R_GS, b)[q] = gs;
            row(R_PXX, b)[q] = pxx; row(R_PYY, b)[q] = pyy; row(R_PXY, b)[q] = pxy; row(R_PHX, b)[q] = phx; row(R_PHY, b)[q] = phy;
        }
        // ---- terminal stage: X_N carries no cost and no distance rows, only its box ----
        {
            double *PN = Pall + (long long)N * ns * ns;
            for (int idx = tid; idx < ns * ns; idx += nt) PN[idx] = 0.0;
            __syncthreads();
            for (int l = tid; l < ns; l += nt) { PN[l * ns + l] = row(R_DGV, N)[l]; row(R_LIN, N)[l] = row(R_GX, N)[l]; }
        }
        __syncthreads();
        NMPC_PROF(0);
        const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
        for (int k = N - 1; k >= 0; k--) {
            const double *Pn = Pall + (long long)(k + 1) * ns * ns;
            double *Pk = Pall + (long long)k * ns * ns, *Yk = Yall + (long long)k * nc * ldy, *Lk = Lall + (long long)k * ncp * ncp;
            double *const Bm = Yk;   // [M_ux | m_u] is assembled in the place of Y_k: it is consumed (bulk copy into shared memory) before Y_k is written back,
                                     // and a separate buffer would cost 200 KB of L2 footprint and of DRAM write-back per stage
            const double *cf = row(R_COEF, k), *cf2 = row(R_COEF2, k);
            const int lds = ncp + 4;   // shared-memory leading dimension of M_uu / L: 4 mod 16, so the 8 x 4 DMMA fragment loads are conflict-free
            // A. pr = p_{k+1} - P_{k+1} rc_{k+1}   (one warp per row)
            {
                const double *rcn = row(R_RC, k + 1), *pn = row(R_LIN, k + 1);
                for (int r0 = wid; r0 < ns; r0 += 4 * nw) {   // four rows per warp at a time: four times the loads in flight
                    double acc[4] = {0.0, 0.0, 0.0, 0.0};
                    for (int j = lane; j < ns; j += 32) {
                        const double v = rcn[j];
#pragma unroll
                        for (int q = 0; q < 4; q++) { const int r = r0 + q * nw; if (r < ns) acc[q] += Pn[r * ns + j] * v; }
                    }
#pragma unroll
                    for (int q = 0; q < 4; q++) {
#pragma unroll
                        for (int m = 16; m > 0; m >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], m);
                        const int r = r0 + q * nw;
                        if (lane == 0 && r < ns) prv[r] = pn[r] - acc[q];
                    }
                }
            }
            // per-robot sums of the condensed collision blocks (curvature and gradient), one (array, robot) per thread: consecutive
            // lanes are consecutive robots, so the gathers of a warp fall into few sectors (a warp-per-sum variant with the partners
            // spread over the lanes was measured twice as slow: its gathers are strided)
            {
                double *dsum = sm + SM_DS;
                for (int idx = tid; idx < 5 * Nr; idx += nt) {
                    const int c = idx / Nr, i = idx - c * Nr;
                    const double *arr = row(R_PXX + c, k + 1);   // R_PXX, R_PYY, R_PXY, R_PHX, R_PHY are consecutive rows
                    double acc = 0.0;
                    for (int jj = 0; jj < i; jj++) { const double v = arr[pairidx(jj, i)]; acc += c >= 3 ? -v : v; }
                    for (int jj = i + 1; jj < Nr; jj++) acc += arr[pairidx(i, jj)];
                    for (int o = 0; o < nobs; o++) acc += arr[Mp + i * nobs + o];   // this robot's static obstacles
                    dsum[idx] = acc;
                }
            }
            __syncthreads();
            NMPC_PROF(1);
            // B. stage matrix M = H~ + [A B]' P+ [A B], one robot pair (i, j) per thread: the 5x5 block C_i' Pb C_j
            for (int idx = tid; idx < Nr * Nr; idx += nt) {
                const int i = idx / Nr, j = idx - i * Nr;
                const double ai = cf[i], bi = cf[Nr + i], tci = cf[2 * Nr + i], tsi = cf[3 * Nr + i];
                const double aj = cf[j], bj = cf[Nr + j], tcj = cf[2 * Nr + j], tsj = cf[3 * Nr + j];
                double t[3][5];
#pragma unroll
                for (int a = 0; a < 3; a++) {
                    const double *pr3 = Pn + (long long)(3 * i + a) * ns + 3 * j;
                    const double p0 = pr3[0], p1 = pr3[1], p2 = pr3[2];
                    t[a][0] = p0; t[a][1] = p1; t[a][2] = p2 + aj * p0 + bj * p1; t[a][3] = tcj * p0 + tsj * p1; t[a][4] = T * p2;
                }
                double G[5][5];
#pragma unroll
                for (int c = 0; c < 5; c++) {
                    G[0][c] = t[0][c]; G[1][c] = t[1][c]; G[2][c] = t[2][c] + ai * t[0][c] + bi * t[1][c];
                    G[3][c] = tci * t[0][c] + tsi * t[1][c]; G[4][c] = T * t[2][c];
                }
                if (i == j) {
                    const double *dgv = row(R_DGV, k), *gxr = row(R_GX, k);
                    G[0][0] += dgv[3 * i]; G[1][1] += dgv[3 * i + 1]; G[2][2] += dgv[3 * i + 2] + cf2[Nr + i];
                    G[3][3] += dgv[ns + 2 * i]; G[4][4] += dgv[ns + 2 * i + 1];
                    G[2][3] += cf2[i]; G[3][2] += cf2[i];
                    const double *dsum = sm + SM_DS;
                    const double sxx = dsum[i], syy = dsum[Nr + i], sxy = dsum[2 * Nr + i], glx = dsum[3 * Nr + i], gly = dsum[4 * Nr + i];
                    G[0][0] += sxx; G[1][1] += syy; G[0][1] += sxy; G[1][0] += sxy;
                    // m = [A B]' pr + h
                    const double p0 = prv[3 * i], p1 = prv[3 * i + 1], p2 = prv[3 * i + 2];
                    row(R_LIN, k)[3 * i] = p0 + gxr[3 * i] + glx;
                    row(R_LIN, k)[3 * i + 1] = p1 + gxr[3 * i + 1] + gly;
                    row(R_LIN, k)[3 * i + 2] = p2 + ai * p0 + bi * p1 + gxr[3 * i + 2];
                    Bm[(long long)(2 * i) * ldy + ns] = tci * p0 + tsi * p1 + gxr[ns + 2 * i];
                    Bm[(long long)(2 * i + 1) * ldy + ns] = T * p2 + gxr[ns + 2 * i + 1];
                } else {
                    const int q = i < j ? pairidx(i, j) : pairidx(j, i);
                    const double vxx = row(R_PXX, k + 1)[q], vyy = row(R_PYY, k + 1)[q], vxy = row(R_PXY, k + 1)[q];
                    G[0][0] -= vxx; G[1][1] -= vyy; G[0][1] -= vxy; G[1][0] -= vxy;
                }
#pragma unroll
                for (int a = 0; a < 3; a++)
#pragma unroll
                    for (int c = 0; c < 3; c++) Pk[(long long)(3 * i + a) * ns + 3 * j + c] = G[a][c];
#pragma unroll
                for (int a = 0; a < 2; a++) {
#pragma unroll
                    for (int c = 0; c < 3; c++) Bm[(long long)(2 * i + a) * ldy + 3 * j + c] = G[3 + a][c];
#pragma unroll
                    for (int c = 0; c < 2; c++) Muu[(2 * i + a) * lds + 2 * j + c] = G[3 + a][3 + c];
                }
            }
            for (int e = nc * ncp + tid; e < ncp * ncp; e += nt) { const int r = e / ncp, c = e - r * ncp; Muu[r * lds + c] = r == c ? 1.0 : 0.0; }   // identity padding up to a multiple of 32
            __syncthreads();
            NMPC_PROF(2);
            // C. blocked right-looking Cholesky M_uu = L L', in place in shared memory (lower triangle, leading dimension lds), by
            //    32-column panels: (1) warp 0 factors the 32 x 32 diagonal block in registers (lane = row, pivot rows exchanged by
            //    shuffles: no CTA barrier inside a panel); (2) one thread per row below it solves x L11' = a by substitution
            //    (L11 broadcast from shared memory); (3) the trailing matrix takes its rank-32 update as 8 x 8 tiles on the FP64
            //    tensor instruction.  Three CTA barriers per panel instead of one per column.  Pivot <= 0: wrong inertia.
            double *Ls = Muu;
            {
                const int g4 = lane >> 2, t4 = lane & 3;
                const int nc8 = (nc + 7) >> 3;   // 8-row tiles that hold rows of M_uu
                for (int j0 = 0; j0 < nc; j0 += 32) {
                    if (wid == 0) {
                        double a[32];
                        double *rp = Ls + (j0 + lane) * lds + j0;
#pragma unroll
                        for (int c = 0; c < 32; c++) a[c] = rp[c];
                        double myrinv = 1.0;
                        bool ok = true;
                        // One straight-line block (a bad pivot only clears `ok`; the NaNs it produces are discarded): step j first brings
                        // column j + 1 up to date and starts its reciprocal square root, then applies the other 30 - j updates of
                        // column j underneath that latency.
                        double d = __shfl_sync(0xffffffffu, a[0], 0);
                        ok = d > 0.0 && d < NMPC_INF;
                        double rinv = wp::rsqrt_pos(d);
                        double *cb = colb + 32;   // two 32-entry column buffers (colb .. colb + 3 ncp is scratch here: the reciprocal diagonals sit in colb[0 .. 31])
#pragma unroll
                        for (int j = 0; j < 32; j++) {
                            const double lij = a[j] * rinv;   // L[lane][j], meaningful for lane >= j
                            a[j] = lij;
                            if (lane == j) myrinv = rinv;
                            double *cj = cb + (j & 1) * 32;
                            cj[lane] = lij;                   // column j for everybody: shuffles would cost two issue slots per entry
                            if (j + 1 < 32) {
                                a[j + 1] = fma(-lij, __shfl_sync(0xffffffffu, lij, j + 1), a[j + 1]);   // the critical entry does not wait for shared memory
                                d = __shfl_sync(0xffffffffu, a[j + 1], j + 1);
                                ok = ok && d > 0.0 && d < NMPC_INF;   // uniform: every lane holds the same value
                                rinv = wp::rsqrt_pos(d);
                            }
                            __syncwarp();
#pragma unroll
                            for (int c = j + 2; c < 32; c++) a[c] = fma(-lij, cj[c], a[c]);   // meaningful for lane >= c
                        }
                        if (ok) {
#pragma unroll
                            for (int c = 0; c < 32; c++)
                                if (c <= lane) rp[c] = a[c];
                            colb[lane] = myrinv;
                        }
                        if (lane == 0) sm[SM_MISC + 3] = ok ? 1.0 : 0.0;
                    }
                    __syncthreads();
                    NMPC_PROF(8);
                    if (sm[SM_MISC + 3] == 0.0) return false;   // uniform
                    // (2) rows below the diagonal block: x <- x L11^-T, right-looking so that the 31 updates of a step are independent
                    {
                        const int r = j0 + 32 + tid;
                        if (r < nc) {
                            double x[32];
                            double *rp = Ls + r * lds + j0;
                            const double *l11 = Ls + j0 * lds + j0;
#pragma unroll
                            for (int c = 0; c < 32; c++) x[c] = rp[c];
#pragma unroll
                            for (int c = 0; c < 32; c++) {
                                x[c] *= colb[c];
#pragma unroll
                                for (int c2 = c + 1; c2 < 32; c2++) x[c2] = fma(-x[c], l11[c2 * lds + c], x[c2]);
                            }
#pragma unroll
                            for (int c = 0; c < 32; c++) rp[c] = x[c];
                        }
                    }
                    __syncthreads();
                    NMPC_PROF(9);
                    // (3) trailing update A22 -= L21 L21' on the lower 8 x 8 tiles: unit = one tile row x up to four tile columns
                    {
                        const int t0 = (j0 >> 3) + 4;
                        int cnt = 0;
                        for (int ti = t0; ti < nc8; ti++)
                            for (int tj0 = t0; tj0 <= ti; tj0 += 4, cnt++) {
                                if (cnt % nw != wid) continue;
                                double acc[4][2];
                                double *cp = Ls + (8 * ti + g4) * lds + 8 * tj0 + 2 * t4;
#pragma unroll
                                for (int q = 0; q < 4; q++) {
                                    const double2 v = tj0 + q <= ti ? *reinterpret_cast<const double2 *>(cp + 8 * q) : make_double2(0.0, 0.0);
                                    acc[q][0] = v.x; acc[q][1] = v.y;
                                }
                                const double *la = Ls + (8 * ti + g4) * lds + j0 + t4, *lb = Ls + (8 * tj0 + g4) * lds + j0 + t4;
#pragma unroll
                                for (int s4 = 0; s4 < 8; s4++) {
                                    const double av = -la[4 * s4];
#pragma unroll
                                    for (int q = 0; q < 4; q++) {
                                        const double bv = tj0 + q <= ti ? lb[8 * q * lds + 4 * s4] : 0.0;
                                        dmma(acc[q], av, bv);
                                    }
                                }
#pragma unroll
                                for (int q = 0; q < 4; q++)
                                    if (tj0 + q <= ti) *reinterpret_cast<double2 *>(cp + 8 * q) = make_double2(acc[q][0], acc[q][1]);
                            }
                    }
                    __syncthreads();
                    NMPC_PROF(10);
                }
            }
            // inverses of the 32 x 32 diagonal blocks of L (one warp per block, one column per lane), stored transposed in
            // the unused upper triangle of the block; reciprocal diagonal in dinv
            {
                const int nblk = ncp >> 5;
                if (wid < nblk) {
                    const int o = wid * 32;
                    double x[32];
                    const int nb_ = nc - o < 32 ? nc - o : 32;   // rows of this block that exist (the padding is an identity)
#pragma unroll
                    for (int i = 0; i < 32; i++) {
                        double acc = i == lane ? 1.0 : 0.0;
                        if (i < nb_) {
#pragma unroll
                            for (int jj = 0; jj < i; jj++) acc -= Ls[(o + i) * lds + o + jj] * x[jj];   // x[jj] = 0 for jj < lane
                            x[i] = i >= lane ? acc / Ls[(o + i) * lds + o + i] : 0.0;
                        } else x[i] = acc;
                    }
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 32; i++) {
                        if (i > lane) Ls[(o + lane) * lds + o + i] = x[i];   // Linv[i][lane], transposed into the upper triangle
                        if (i == lane) dinv[o + lane] = x[i];
                    }
                }
            }
            __syncthreads();
            for (int e = tid; e < ncp * ncp; e += nt) { const int r = e / ncp, c = e - r * ncp; Lk[e] = Ls[r * lds + c]; }   // kept for the forward pass (lower triangle), leading dimension ncp in global memory
            // W_IJ = Linv_II L_IJ for the blocks below the diagonal (I > J), while L is still in shared memory: with V = blockdiag(Linv) B
            // the forward substitution becomes Y_I = V_I - sum_{J < I} W_IJ Y_J, one contraction and one barrier per block row instead of
            // a contraction, a barrier, a triangular product and two more barriers.  W goes to the CTA's scratch (A fragments later).
            {
                const int g4 = lane >> 2, t4 = lane & 3, nblk = ncp >> 5;
                const int nunit = 2 * nblk * (nblk - 1);   // (block pair, tile row)
                for (int unit = wid; unit < nunit; unit += nw) {
                    const int ta = (unit + (unit >> 2)) & 3, bp = unit >> 2;
                    int I = 1;
                    while ((I + 1) * I / 2 <= bp) I++;
                    const int J = bp - I * (I - 1) / 2;
                    const int rl = 8 * ta + g4;
                    double acc[4][2];
#pragma unroll
                    for (int q = 0; q < 4; q++) { acc[q][0] = 0.0; acc[q][1] = 0.0; }
                    const double *lb = Ls + (32 * I + t4) * lds + 32 * J + g4;   // B fragment: L[32 I + 4 s + t4][32 J + 8 q + g4]
                    for (int s4 = 0; s4 < 2 * ta + 2; s4++) {
                        const int u = 4 * s4 + t4;
                        const double a = u < rl ? Ls[(32 * I + u) * lds + 32 * I + rl] : (u == rl ? dinv[32 * I + rl] : 0.0);
#pragma unroll
                        for (int q = 0; q < 4; q++) dmma(acc[q], a, lb[4 * s4 * lds + 8 * q]);
                    }
                    double *wp_ = Wg + (long long)bp * 1024 + rl * 32 + 2 * t4;
#pragma unroll
                    for (int q = 0; q < 4; q++) *reinterpret_cast<double2 *>(wp_ + 8 * q) = make_double2(acc[q][0], acc[q][1]);
                }
            }
            NMPC_PROF(3);
            // D. Y = L^-1 [M_ux | m_u] with Y resident in shared memory (it stays there for the rank-k update): blocked forward
            //    substitution over 32-row blocks on the FP64 tensor instruction (mma.sync m8n8k4, see dmma()).  A unit of work is one
            //    8-row tile row of the block times four 8-column tiles; its accumulators stay in registers over the whole
            //    contraction.  L (and the inverses of its diagonal blocks, stored transposed in the upper triangles) is read back
            //    from global memory as A fragments; the B fragments come from the rows of Y that are already final.
            __syncthreads();   // Ls has been copied to Lk by every thread: its shared memory now becomes Y
            double *Ys = Muu;
            const int nt8 = (ns + 1 + 7) >> 3;   // 8-column tiles of [Y | y_m]
            const int g4 = lane >> 2, t4 = lane & 3;
            {
                const double *Lg = Lk;
                // [M_ux | m_u] (written by the build step with ordinary stores) comes in as ONE bulk copy (TMA, completion on the CTA's
                // mbarrier): a thread-strided copy loop spent 10-18 k cycles per stage on L2 / DRAM round trips
                if (tid == 0) {
                    asm volatile("fence.proxy.async;" ::: "memory");
                    const unsigned bytes = (unsigned)(nc * ldy) * 8u;
                    wp::bulk_expect(sm + SM_MBAR, bytes);
                    wp::bulk_g2s(Ys, Bm, bytes, sm + SM_MBAR);
                }
                for (int e = nc * ldy + tid; e < ((nc + 3) & ~3) * ldy; e += nt) Ys[e] = 0.0;   // rows up to a multiple of four: zero (k-steps of the rank-k update)
                wp::mbar_wait(sm + SM_MBAR, bar_phase);
                bar_phase ^= 1u;
                __syncthreads();
                NMPC_PROF(11);
                const int nblk = ncp >> 5, ngrp = (nt8 + 3) >> 2;
                // V = blockdiag(Linv_II) B in place.  Unit = (block row I, group of four tile columns); the warp walks the four tile
                // rows from the bottom up: tile row ta reads rows <= 8 ta + 7 of the block and writes its own, so the rows it leaves
                // behind are still the original B.  Linv_II[i][u] (u < i) sits at L[32 I + u][32 I + i], its diagonal in dinv.
                for (int unit = wid; unit < nblk * ngrp; unit += nw) {
                    const int I = unit % nblk, j0 = 4 * (unit / nblk);
                    double al[4][8];
#pragma unroll
                    for (int ta = 0; ta < 4; ta++)
#pragma unroll
                        for (int s4 = 0; s4 < 8; s4++) {
                            const int rl = 8 * ta + g4, u = 4 * s4 + t4;
                            al[ta][s4] = s4 < 2 * ta + 2 ? (u < rl ? Lg[(long long)(32 * I + u) * ncp + 32 * I + rl] : (u == rl ? dinv[32 * I + rl] : 0.0)) : 0.0;
                        }
                    const double *yb = Ys + (32 * I + t4) * ldy + 8 * j0 + g4;
#pragma unroll
                    for (int ta = 3; ta >= 0; ta--) {
                        if (32 * I + 8 * ta >= nc) continue;   // warp-uniform: no rows of Y in this tile row
                        const int r = 32 * I + 8 * ta + g4;
                        double acc[4][2];
#pragma unroll
                        for (int q = 0; q < 4; q++) { acc[q][0] = 0.0; acc[q][1] = 0.0; }
#pragma unroll
                        for (int s4 = 0; s4 < 8; s4++) {
                            if (s4 < 2 * ta + 2) {
                                const bool rowok = 32 * I + 4 * s4 + t4 < nc;
#pragma unroll
                                for (int q = 0; q < 4; q++) {
                                    const double b = rowok && j0 + q < nt8 ? yb[4 * s4 * ldy + 8 * q] : 0.0;
                                    dmma(acc[q], al[ta][s4], b);
                                }
                            }
                        }
#pragma unroll
                        for (int q = 0; q < 4; q++) {
                            const int cc = 8 * (j0 + q) + 2 * t4;
                            if (r < nc && j0 + q < nt8 && cc < ldy)
                                *reinterpret_cast<double2 *>(Ys + r * ldy + cc) = make_double2(acc[q][0], acc[q][1]);
                        }
                    }
                }
                __syncthreads();
                NMPC_PROF(12);
                // Y_I = V_I - sum_{J < I} W_IJ Y_J, block row by block row.  warp -> (tile row, column groups): the four warps
                // wid = 4 h .. 4 h + 3 take the four tile rows of the column groups g = h, h + nw / 4 (ngrp <= nw / 2 for every Nr).  The
                // A fragments -W[r][.] do not depend on Y: all of them are requested at once (one L2 round trip per block row).
                const int ta = (wid + (wid >> 2)) & 3, gh = wid >> 2, gstep = nw >> 2;
                for (int I = 1; I < nblk; I++) {
                    const int r = 32 * I + 8 * ta + g4;   // this thread's row of the C fragments
                    if (32 * I + 8 * ta < nc) {           // warp-uniform
                        double af[24];
                        const double *wa = Wg + (long long)(I * (I - 1) / 2) * 1024 + (8 * ta + g4) * 32 + t4;
#pragma unroll
                        for (int s4 = 0; s4 < 24; s4++) af[s4] = s4 < 8 * I ? -wa[(s4 >> 3) * 1024 + 4 * (s4 & 7)] : 0.0;
#pragma unroll
                        for (int rd = 0; rd < 2; rd++) {
                            const int g = gh + rd * gstep, j0 = 4 * g;
                            if (g >= ngrp) continue;   // warp-uniform
                            double c1[4][2];
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                const int cc = 8 * (j0 + q) + 2 * t4;
                                const bool ok = r < nc && j0 + q < nt8 && cc < ldy;
                                const double2 v = ok ? *reinterpret_cast<const double2 *>(Ys + r * ldy + cc) : make_double2(0.0, 0.0);
                                c1[q][0] = v.x; c1[q][1] = v.y;
                            }
                            const double *yb = Ys + t4 * ldy + 8 * j0 + g4;   // B fragment: Y[4 s + t4][8 (j0 + q) + g4]
#pragma unroll
                            for (int s4 = 0; s4 < 24; s4++) {
                                if (s4 < 8 * I) {
#pragma unroll
                                    for (int q = 0; q < 4; q++) {
                                        const double b = j0 + q < nt8 ? yb[4 * s4 * ldy + 8 * q] : 0.0;
                                        dmma(c1[q], af[s4], b);
                                    }
                                }
                            }
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                const int cc = 8 * (j0 + q) + 2 * t4;
                                if (r < nc && j0 + q < nt8 && cc < ldy)
                                    *reinterpret_cast<double2 *>(Ys + r * ldy + cc) = make_double2(c1[q][0], c1[q][1]);
                            }
                        }
                    }
                    __syncthreads();
                }
                NMPC_PROF(13);
                for (int e = tid; e < nc * (ldy / 2); e += nt)   // kept for the forward pass
                    reinterpret_cast<double2 *>(Yk)[e] = reinterpret_cast<const double2 *>(Ys)[e];
            }
            NMPC_PROF(4);
            // F. [P_k | p_k] = [M_xx | m_x] - Y' [Y | y_m]: the upper 8 x 8 tiles of the Gram matrix of the resident Y on the FP64 tensor
            //    instruction, one tile row times four tile columns per unit (A fragment shared by the four), mirrored on the store
            {
                int cnt = 0;
                const int nk4 = (nc + 3) >> 2;
                for (int ti = 0; ti < nt8; ti++)
                    for (int j0 = ti; j0 < nt8; j0 += 4, cnt++) {
                        if (cnt % nw != wid) continue;
                        const int r = 8 * ti + g4;
                        double acc[4][2], pv[4][2];
#pragma unroll
                        for (int q = 0; q < 4; q++)
#pragma unroll
                            for (int e = 0; e < 2; e++) {   // M_xx tile: issued before the contraction so that its latency overlaps
                                const int cc = 8 * (j0 + q) + 2 * t4 + e;
                                acc[q][e] = 0.0;
                                pv[q][e] = (r < ns && cc < ns && r <= cc) ? Pk[(long long)r * ns + cc] : 0.0;
                            }
                        const double *ya = Ys + t4 * ldy + 8 * ti + g4, *yb = Ys + t4 * ldy + 8 * j0 + g4;
#pragma unroll 4
                        for (int s4 = 0; s4 < nk4; s4++) {
                            const double a = ya[4 * s4 * ldy];
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                const double b = j0 + q < nt8 ? yb[4 * s4 * ldy + 8 * q] : 0.0;
                                dmma(acc[q], a, b);
                            }
                        }
#pragma unroll
                        for (int q = 0; q < 4; q++)
#pragma unroll
                            for (int e = 0; e < 2; e++) {
                                const int cc = 8 * (j0 + q) + 2 * t4 + e;
                                if (r < ns && cc < ns && r <= cc) {
                                    const double v = pv[q][e] - acc[q][e];
                                    Pk[(long long)r * ns + cc] = v; Pk[(long long)cc * ns + r] = v;
                                } else if (r < ns && cc == ns) row(R_LIN, k)[r] -= acc[q][e];
                            }
                    }
            }
            __syncthreads();
            NMPC_PROF(5);
        }
        return true;
    }

    // ---------------------------------------------------------------------------------------
    // forward pass: steps, new multipliers, fraction-to-boundary step sizes, grad(phi)'d
    // ---------------------------------------------------------------------------------------
    NMPC_BPASS void forward(double mu, double tau, int rdz, int rds, int rytc, int rytd, StepInfo &si)
    {
        NMPC_BLK_LOCALS
        double ap = 0.0, az = 0.0, gbd = 0.0, tiny = 0.0;
        NMPC_PROF_BEGIN
        double *dzb = sm + SM_DZB, *dxn = sm + SM_DXN, *tb = sm + SM_TB, *xb = sm + SM_XB, *Ls = sm + SM_MUU;
        const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
        __syncthreads();
        for (int q = tid; q < M; q += nt) {
            const double rd = row(R_RD, 0)[q], Dq = row(R_DQ, 0)[q], gs = row(R_GS, 0)[q];
            const bool act = DL[q] > -NMPC_INF || DU[q] < NMPC_INF;
            const double ds = act ? rd : 0.0, ytd = act ? Dq * ds + gs : 0.0;
            row(rds, 0)[q] = ds; row(rytd, 0)[q] = ytd;
            if (act) {
                const double s = row(R_S, 0)[q];
                WS::slack_step_terms(s, ds, DL[q], DU[q], row(R_VL, 0)[q], row(R_VU, 0)[q], mu, ap, az);
                gbd += gs * ds; tiny = fmax(tiny, fabs(ds) / (1.0 + fabs(s)));
            }
        }
        for (int l = tid; l < nz; l += nt) dzb[l] = l < ns ? -row(R_RC, 0)[l] : 0.0;
        __syncthreads();
        for (int k = 0; k <= N; k++) {
            const double *Pk = Pall + (long long)k * ns * ns;
            const double *Yk = Yall + (long long)(k < N ? k : 0) * nc * ldy, *Lk = Lall + (long long)(k < N ? k : 0) * ncp * ncp;
            // the stage's Cholesky factor comes into shared memory as one bulk copy (TMA) underneath the mat-vecs below: the back
            // substitution is a chain of dependent reads, which out of global memory cost an L2 / DRAM round trip per link
            if (k < N && tid == 0) {
                asm volatile("fence.proxy.async;" ::: "memory");
                const unsigned bytes = (unsigned)(ncp * ncp) * 8u;
                wp::bulk_expect(sm + SM_MBAR, bytes);
                wp::bulk_g2s(Ls, Lk, bytes, sm + SM_MBAR);
            }
            // y~c_k = -(P_k dx + p_k);  t = Y_k dx + y_m      (one warp per row)
            const int nrows = ns + (k < N ? nc : 0);
            for (int r0 = wid; r0 < nrows; r0 += 4 * nw) {   // four rows per warp at a time
                const double *mr[4];
                double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const int r = r0 + q * nw < nrows ? r0 + q * nw : r0;
                    mr[q] = r < ns ? Pk + (long long)r * ns : Yk + (long long)(r - ns) * ldy;
                }
                for (int j = lane; j < ns; j += 32) {
                    const double v = dzb[j];
#pragma unroll
                    for (int q = 0; q < 4; q++) acc[q] += mr[q][j] * v;
                }
#pragma unroll
                for (int q = 0; q < 4; q++) {
#pragma unroll
                    for (int m = 16; m > 0; m >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], m);
                    const int r = r0 + q * nw;
                    if (lane == 0 && r < nrows) {
                        if (r < ns) row(rytc, k)[r] = -(acc[q] + row(R_LIN, k)[r]);
                        else tb[r - ns] = acc[q] + mr[q][ns];
                    }
                }
            }
            __syncthreads();
            if (k < N) {   // L' x = t by 32-row blocks: x_I = Linv_II' (t_I - sum_{J > I} L_JI' x_J), du = -x.  L is read from its
                           // shared-memory image (leading dimension ncp); Linv_II sits transposed in the upper triangle of block (I, I)
                wp::mbar_wait(sm + SM_MBAR, bar_phase);
                bar_phase ^= 1u;
                double *red = Ls + ncp * ncp;   // nw x 32 partial sums (ncp (ncp + 4) doubles are reserved: 4 ncp = 32 nw)
                for (int I = (ncp >> 5) - 1; I >= 0; I--) {
                    const int i = lane, gi = 32 * I + lane;
                    double part = 0.0;
                    for (int u = 32 * (I + 1) + wid; u < nc; u += nw) part += Ls[u * ncp + gi] * xb[u];
                    red[wid * 32 + i] = part;
                    __syncthreads();
                    if (wid == 0) {
                        double ti = gi < nc ? tb[gi] : 0.0;
                        for (int w = 0; w < nw; w++) ti -= red[w * 32 + i];
                        double acc = ti / Ls[gi * ncp + gi];
                        const int nb_ = nc - 32 * I < 32 ? nc - 32 * I : 32;   // rows of this block that exist
#pragma unroll 8
                        for (int u = 1; u < nb_; u++) {
                            const double tu = __shfl_sync(0xffffffffu, ti, u);
                            const double lv = u > i ? Ls[gi * ncp + 32 * I + u] : 0.0;
                            acc += lv * tu;
                        }
                        if (gi < nc) xb[gi] = acc;
                    }
                    __syncthreads();
                }
                for (int u = tid; u < nc; u += nt) dzb[ns + u] = -xb[u];
            } else {
                for (int u = tid; u < nc; u += nt) dzb[ns + u] = 0.0;
            }
            __syncthreads();
            for (int l = tid; l < nz; l += nt) {
                const double dzl = dzb[l];
                row(rdz, k)[l] = dzl;
                if (l < nvalid(k)) {
                    const double z = row(R_Z, k)[l];
                    WS::slack_step_terms(z, dzl, BL[k * W + l], BU[k * W + l], row(R_ZL, k)[l], row(R_ZU, k)[l], mu, ap, az);
                    gbd += row(R_GX, k)[l] * dzl; tiny = fmax(tiny, fabs(dzl) / (1.0 + fabs(z)));
                }
            }
            if (k < N) {
                const double *cf = row(R_COEF, k);
                for (int l = tid; l < ns; l += nt) {
                    const int rob = l / 3, comp = l - 3 * rob;
                    const double cA = comp == 0 ? cf[rob] : (comp == 1 ? cf[Nr + rob] : 0.0);
                    const double cB = comp == 0 ? cf[2 * Nr + rob] : (comp == 1 ? cf[3 * Nr + rob] : T);
                    dxn[l] = dzb[l] + cA * dzb[3 * rob + 2] + cB * dzb[ns + 2 * rob + (comp == 2 ? 1 : 0)] - row(R_RC, k + 1)[l];
                }
                const int b = k + 1;
                for (int q = tid; q < M; q += nt) {
                    // (all loads of the row before the branch on its bounds, see eval)
                    const double lo = DL[b * W + q], hi = DU[b * W + q];
                    const double gs = row(R_GS, b)[q], gxq_ = row(R_GXQ, b)[q], gyq_ = row(R_GYQ, b)[q], rd_ = row(R_RD, b)[q], dq_ = row(R_DQ, b)[q];
                    const double s = row(R_S, b)[q], vl_ = row(R_VL, b)[q], vu_ = row(R_VU, b)[q];
                    double ddx, ddy;
                    if (q < Mp) { const int pi = pairs[2 * q], pj = pairs[2 * q + 1]; ddx = dzb[3 * pi] - dzb[3 * pj]; ddy = dzb[3 * pi + 1] - dzb[3 * pj + 1]; }
                    else { const int pi = (q - Mp) / nobs; ddx = dzb[3 * pi]; ddy = dzb[3 * pi + 1]; }
                    const bool act = lo > -NMPC_INF || hi < NMPC_INF;
                    double ds = 0.0, ytd = 0.0;
                    if (act) {
                        ds = gxq_ * ddx + gyq_ * ddy + rd_;
                        ytd = dq_ * ds + gs;
                        WS::slack_step_terms(s, ds, lo, hi, vl_, vu_, mu, ap, az);
                        gbd += gs * ds; tiny = fmax(tiny, fabs(ds) / (1.0 + fabs(s)));
                    }
                    row(rds, b)[q] = ds; row(rytd, b)[q] = ytd;
                }
                __syncthreads();
                for (int l = tid; l < nz; l += nt) dzb[l] = l < ns ? dxn[l] : 0.0;
            }
            __syncthreads();
        }
        double v[4] = {ap, az, gbd, tiny};
        NMPC_PROF(6);
        breduce<4>(v, 0xBu);   // ap, az, tiny are maxima; gbd a sum
        si.ap = v[0] > tau ? tau / v[0] : 1.0; si.az = v[1] > tau ? tau / v[1] : 1.0;
        si.gbd = v[2]; si.tiny = v[3];
    }

    // ---------------------------------------------------------------------------------------
    NMPC_BPASS void accept(double alpha, double az, double mu, int rdz, int rds, int rytc, int rytd)
    {
        NMPC_BLK_LOCALS
        const double ks = P.o.kappa_sigma, iks = 1.0 / ks;
        auto mult = [=](double m, double sl_old, double sl_new, double dv_signed) {
            const double r = 1.0 / sl_old, c = mu / sl_new;
            const double m2 = m + az * (mu * r - m + m * r * dv_signed);
            return fmax(fmin(m2, ks * c), iks * c);
        };
        for (int idx = tid; idx < S * W; idx += nt) {
            const int k = idx / W, l = idx - k * W;
            // (all loads of an entry before the branches on its bounds, see eval)
            if (l < nvalid(k)) {
                const double z = row(R_Z, k)[l], dz = row(rdz, k)[l], lo = BL[k * W + l], hi = BU[k * W + l];
                const double zl_ = row(R_ZL, k)[l], zu_ = row(R_ZU, k)[l];
                const double zn = z + alpha * dz;
                if (lo > -NMPC_INF) row(R_ZL, k)[l] = mult(zl_, z - lo, zn - lo, -dz);
                if (hi < NMPC_INF) row(R_ZU, k)[l] = mult(zu_, hi - z, hi - zn, dz);
                row(R_Z, k)[l] = zn;
            }
            if (l < ns) { const double yc = row(R_YC, k)[l]; row(R_YC, k)[l] = yc + alpha * (row(rytc, k)[l] - yc); }
            if (l < M) {
                const double lo = DL[k * W + l], hi = DU[k * W + l];
                const double s = row(R_S, k)[l], ds = row(rds, k)[l], vl_ = row(R_VL, k)[l], vu_ = row(R_VU, k)[l];
                const double yd = row(R_YD, k)[l], ytd_ = row(rytd, k)[l];
                if (lo > -NMPC_INF || hi < NMPC_INF) {
                    const double sn_ = s + alpha * ds;
                    if (lo > -NMPC_INF) row(R_VL, k)[l] = mult(vl_, s - lo, sn_ - lo, -ds);
                    if (hi < NMPC_INF) row(R_VU, k)[l] = mult(vu_, hi - s, hi - sn_, ds);
                    row(R_S, k)[l] = sn_;
                    row(R_YD, k)[l] = yd + alpha * (ytd_ - yd);
                }
            }
        }
        __syncthreads();
    }

    NMPC_BPASS void accept_primal(double alpha, int rdz, int rds)
    {
        NMPC_BLK_LOCALS
        for (int idx = tid; idx < S * W; idx += nt) {
            const int k = idx / W, l = idx - k * W;
            if (l < nvalid(k)) row(R_Z, k)[l] += alpha * row(rdz, k)[l];
            if (l < M && (DL[k * W + l] > -NMPC_INF || DU[k * W + l] < NMPC_INF)) row(R_S, k)[l] += alpha * row(rds, k)[l];
        }
        __syncthreads();
    }

    // after the restoration fallback: equality multipliers reset, bound multipliers clipped
    NMPC_BPASS void resto_reset(double mu)
    {
        NMPC_BLK_LOCALS
        const double ks = P.o.kappa_sigma;
        for (int idx = tid; idx < S * W; idx += nt) {
            const int k = idx / W, l = idx - k * W;
            if (l < nvalid(k)) {
                const double z = row(R_Z, k)[l], lo = BL[k * W + l], hi = BU[k * W + l];
                if (lo > -NMPC_INF) { const double s2 = z - lo; row(R_ZL, k)[l] = fmax(fmin(row(R_ZL, k)[l], ks * mu / s2), mu / (ks * s2)); }
                if (hi < NMPC_INF) { const double s2 = hi - z; row(R_ZU, k)[l] = fmax(fmin(row(R_ZU, k)[l], ks * mu / s2), mu / (ks * s2)); }
            }
            row(R_YC, k)[l] = 0.0; row(R_YD, k)[l] = 0.0;
            if (l < M) {
                const double s = row(R_S, k)[l], lo = DL[k * W + l], hi = DU[k * W + l];
                if (lo > -NMPC_INF) { const double s2 = s - lo; row(R_VL, k)[l] = fmax(fmin(row(R_VL, k)[l], ks * mu / s2), mu / (ks * s2)); }
                if (hi < NMPC_INF) { const double s2 = hi - s; row(R_VU, k)[l] = fmax(fmin(row(R_VU, k)[l], ks * mu / s2), mu / (ks * s2)); }
            }
        }
        __syncthreads();
    }

    // restoration candidate: forward rollout of the current controls, slacks reset from the distances;
    // written as a direction (R_DZ, R_DS) = candidate - iterate
    NMPC_BPASS void rollout_project()
    {
        NMPC_BLK_LOCALS
        const nmpc_opts &o = P.o;
        double *zt = sm + SM_DZB, *zn = sm + SM_TB /* ns <= nc + nc + ... : see below */, *cs = sm + SM_CS;
        // zn needs ns doubles: SM_TB (nc) and SM_XB (nc) are contiguous, 2 nc = 4 Nr >= 3 Nr
        __syncthreads();
        for (int l = tid; l < nz; l += nt)
            zt[l] = l < ns ? WS::push_in(pp[l] + CE[l], BL[l], BU[l], o.bound_push, o.bound_frac) : row(R_Z, 0)[l];
        __syncthreads();
        for (int k = 0; k <= N; k++) {
            for (int l = tid; l < nz; l += nt) row(R_DZ, k)[l] = l < nvalid(k) ? zt[l] - row(R_Z, k)[l] : 0.0;
            if (k < N) for (int i = tid; i < Nr; i += nt) { double s_, c_; sincos(zt[3 * i + 2], &s_, &c_); cs[i] = c_; cs[Nr + i] = s_; }
            for (int q = tid; q < M; q += nt) {
                for (int pass = (k == 0 ? 0 : 1); pass < 2; pass++) {
                    if (pass == 1 && k == N) break;
                    const int b = pass == 0 ? 0 : k + 1;
                    const double lo = DL[b * W + q], hi = DU[b * W + q];
                    double dv = NMPC_DUMMY_ROW_VALUE;
                    if (pass == 1) dv = rowgeom(zt, q, Mp, nobs, pairs, obs + k * ostr).dv;
                    const bool act = lo > -NMPC_INF || hi < NMPC_INF;
                    row(R_DS, b)[q] = act ? WS::push_in(dv, lo, hi, o.bound_push, o.bound_frac) - row(R_S, b)[q] : 0.0;
                }
            }
            __syncthreads();
            if (k < N) {
                for (int l = tid; l < ns; l += nt) {
                    const int rob = l / 3, comp = l - 3 * rob;
                    const double v = zt[ns + 2 * rob];
                    double x = comp == 0 ? zt[l] + T * v * cs[rob] : (comp == 1 ? zt[l] + T * v * cs[Nr + rob] : zt[l] + T * zt[ns + 2 * rob + 1]);
                    zn[l] = WS::push_in(x + CE[(k + 1) * W + l], BL[(k + 1) * W + l], BU[(k + 1) * W + l], o.bound_push, o.bound_frac);
                }
                __syncthreads();
                for (int l = tid; l < nz; l += nt) zt[l] = l < ns ? zn[l] : (k + 1 < N ? row(R_Z, k + 1)[l] : 0.0);
            }
            __syncthreads();
        }
    }

    NMPC_BPASS void soc_begin()
    {
        NMPC_BLK_LOCALS
        for (int idx = tid; idx < S * W; idx += nt) {
            const int k = idx / W, l = idx - k * W;
            row(R_CSOC, k)[l] = l < ns ? row(R_RC, k)[l] : 0.0;
            row(R_DSOC, k)[l] = l < M ? row(R_RD, k)[l] : 0.0;
        }
        __syncthreads();
    }

    __device__ double mult_absmax()
    {
        NMPC_BLK_LOCALS
        double ymax = 0.0;
        for (int idx = tid; idx < S * W; idx += nt) {
            const int k = idx / W, l = idx - k * W;
            if (l < ns) ymax = fmax(ymax, fabs(row(R_YC, k)[l]));
            if (l < M) ymax = fmax(ymax, fabs(row(R_YD, k)[l]));
        }
        return bmax(ymax);
    }
    __device__ void mult_zero()
    {
        NMPC_BLK_LOCALS
        for (int idx = tid; idx < S * W; idx += nt) { const int k = idx / W, l = idx - k * W; row(R_YC, k)[l] = 0.0; row(R_YD, k)[l] = 0.0; }
    }

    // ---------------------------------------------------------------------------------------
    // filter (shared memory; thread 0 edits)
    // ---------------------------------------------------------------------------------------
    // IPOPT's filter is unbounded inside a barrier subproblem: it lives in the slot's global scratch, append-only (an entry
    // that a newer one dominates is redundant for the test and stays); an overflow overwrites the oldest and is counted.
    __device__ double *filter_base() const { return Wg + (long long)((ncp >> 5) * ((ncp >> 5) - 1) / 2) * 1024; }
    __device__ bool filter_ok(double th, double ph) const
    {
        const double *fth = wp::global_ptr(filter_base()), *fph = fth + NMPC_FILTER_CAP;
        const int m = fn < NMPC_FILTER_CAP ? fn : NMPC_FILTER_CAP;
        for (int i = 0; i < m; i++)
            if (!(th < fth[i] || ph < fph[i])) return false;
        return true;
    }
    NMPC_BPASS void filter_add(double th, double ph)
    {
        NMPC_BLK_LOCALS
        double *fth = wp::global_ptr(filter_base()), *fph = fth + NMPC_FILTER_CAP;
        __syncthreads();
        if (tid == 0) {
            const int slot = fn % NMPC_FILTER_CAP;
            fth[slot] = th; fph[slot] = ph;
            if (fn >= NMPC_FILTER_CAP) sm[SM_MISC + 2] += 1.0;
        }
        fn++;
        __syncthreads();
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

    // outputs in the reference layout, multipliers in CasADi's sign convention
    NMPC_BPASS void write_outputs(int st, int iter, double E0, double pinf, double dinf, double c0, double mu)
    {
        NMPC_BLK_LOCALS
        const long long n = (long long)ns * S + (long long)nc * N, mg = goff(N) + ns + M;
        double *x = P.x + inst * n;
        double *lx = P.lam_x ? P.lam_x + inst * n : nullptr;
        double *g = P.g ? P.g + inst * mg : nullptr;
        double *lg = P.lam_g ? P.lam_g + inst * mg : nullptr;
        double fo = 0.0;
        trig_rows(0.0, 0, false, R_TRIG);
        for (int idx = tid; idx < S * nz; idx += nt) {
            const int k = idx / nz, l = idx - k * nz;
            if (l >= nvalid(k)) continue;
            const double zk = row(R_Z, k)[l];
            const long long xi = l < ns ? (long long)k * ns + l : (long long)ns * S + (long long)k * nc + (l - ns);
            x[xi] = zk;
            if (lx) lx[xi] = (row(R_ZU, k)[l] - row(R_ZL, k)[l]) / df;
            if (k < N) { const double e = zk - ref(k, l); fo += 0.5 * qw(l) * e * e; }
        }
        for (int idx = tid; idx < S * ns; idx += nt) {
            const int k = idx / ns, l = idx - k * ns;
            if (g) g[goff(k) + l] = k == 0 ? row(R_Z, 0)[l] - pp[l] : row(R_Z, k)[l] - predict(row(R_Z, k - 1), row(R_TRIG, k - 1), l);
            if (lg) lg[goff(k) + l] = row(R_YC, k)[l] / df;
        }
        for (int idx = tid; idx < S * M; idx += nt) {
            const int b = idx / M, q = idx - b * M;
            if (family && b == 0) continue;   // family 1: block 0 holds the initial condition only
            double dv = NMPC_DUMMY_ROW_VALUE;
            if (b > 0) dv = rowgeom(row(R_Z, b - 1), q, Mp, nobs, pairs, obs + (b - 1) * ostr).dv;
            if (g) g[goff(b) + ns + q] = dv;
            if (lg) lg[goff(b) + ns + q] = row(R_YD, b)[q] / df;
        }
        fo = bsum(fo);
        if (tid == 0) {
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
        __syncthreads();
    }

    __device__ void run() { ipm_run(*this); }
};

// persistent kernel: one CTA per instance, instances pulled from the same atomic queue as the warp kernel
__global__ void __launch_bounds__(NMPC_BLOCK_THREADS, 1) solve_kernel_block(const NmpcSolveParams P)
{
    extern __shared__ double smem[];
    double *ws = P.ws + (long long)blockIdx.x * P.ws_stride;
    BlockSolver s(P, smem, ws);
    __shared__ int next_inst;
    if (threadIdx.x == 0) wp::mbar_init(smem + BlockSolver::SM_MBAR);
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) next_inst = atomicAdd(P.counter, 1);
        __syncthreads();
        const int slot = next_inst;
        if (slot >= P.B) break;
        s.setup(P.order ? P.order[slot] : slot);
        s.run();
    }
}
