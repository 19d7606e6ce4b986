// libnmpc_b200.so -- C-ABI (include/nmpc_b200.h) over the sm_100a kernels.
// No CPU fallback: every entry point launches CUDA work or fails with NMPC_ECUDA.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "nmpc_b200.h"
#include "warp_prims.cuh"
#include "solver_body.cuh"
#include "block_solver.cuh"
#include "small_ocp.cuh"
#include "aux_kernels.cuh"

#define NMPC_OBS_WARP_MAX_ROBOTS 4   // the static-obstacle family is instantiated on the warp path for 1..4 robots
#ifndef SOLVE_WARPS
#define SOLVE_WARPS 4     // warps (instances) per CTA = the convoy group, see WarpSolver::iter_sync
#endif
#ifndef SOLVE_MIN_CTAS
#define SOLVE_MIN_CTAS 3   // 12 resident instances per SM (13.2 KB of shared memory each, <= 168 registers per thread).  Measured
                           // (round 2, profiles/sweeps_r2.md): 4 x 3 -> 46.4 k, 3 x 4 -> 45.1 k, 6 x 2 -> 45.6 k, 2 x 6 -> 43.2 k solves/s;
                           // 128-register builds with 15-16 warps per SM (3 x 5, 4 x 4, 2 x 8) -> 34-35 k: their spills go to
                           // local memory while 16 x 13.2 KB of shared memory leaves almost no L1 to hold them
#endif

static thread_local char g_err[512] = "";
static int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_OK(call)                                                                                    \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) return fail(NMPC_ECUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

extern "C" const char *nmpc_last_error(void) { return g_err; }

extern "C" void nmpc_default_opts(nmpc_opts *o)
{
    o->tol = 1e-8; o->max_iter = 2000; o->acceptable_tol = 1e-8; o->acceptable_iter = 15;
    o->acceptable_obj_change_tol = 1e-6; o->dual_inf_tol = 1.0; o->constr_viol_tol = 1e-4; o->compl_inf_tol = 1e-4;
    o->mu_init = 0.1; o->kappa_mu = 0.2; o->theta_mu = 1.5; o->barrier_tol_factor = 10.0; o->tau_min = 0.99;
    o->bound_push = 0.01; o->bound_frac = 0.01; o->bound_relax_factor = 1e-8; o->bound_mult_init_val = 1.0;
    o->constr_mult_init_max = 1e3; o->kappa_sigma = 1e10; o->kappa_d = 1e-5; o->nlp_scaling_max_gradient = 100.0;
    o->max_soc = 4; o->max_resto_iter = 100;
}

// ------------------------------------------------------------------------------------------------
// the persistent solve kernel: one warp per instance, instances pulled from an atomic queue
// ------------------------------------------------------------------------------------------------
// threads per CTA and instances ("teams") per CTA: one warp per instance up to 6 robots (4 per CTA, 3 CTAs per SM);
// 7..10 robots use the two-warp team (2 per CTA on named barriers, 2 CTAs per SM: 255 registers per thread).  The
// one-warp teams of a CTA are a convoy group (WarpSolver::iter_sync).
template <int NR, bool OBS = false, bool TRK = false> struct SolveCfg {
    static constexpr int LW = WarpSolver<NR, OBS, TRK>::LW;
    static constexpr int THREADS = LW == 32 ? SOLVE_WARPS * 32 : 128;
    static constexpr int TEAMS = THREADS / LW;
    static constexpr int MIN_CTAS = LW == 32 ? SOLVE_MIN_CTAS : 2;
};

// OBS: the static-obstacle family; TRK: trajectory tracking (each its own instantiation, see WarpSolver)
template <int NR, bool OBS = false, bool TRK = false>
__global__ void __launch_bounds__((SolveCfg<NR, OBS, TRK>::THREADS), (SolveCfg<NR, OBS, TRK>::MIN_CTAS)) solve_kernel(const NmpcSolveParams P)
{
    extern __shared__ double smem[];
    typedef WarpSolver<NR, OBS, TRK> WSol;
    constexpr int LW = SolveCfg<NR, OBS, TRK>::LW;
    const int team = threadIdx.x / LW, tl = threadIdx.x & (LW - 1);
    double *sm = smem + (size_t)team * WSol::SM_DOUBLES;
    double *ws = P.ws + ((long long)blockIdx.x * SolveCfg<NR, OBS, TRK>::TEAMS + team) * P.ws_stride;
    WSol s(P, sm, ws);
    s.init_team();
    for (;;) {
        WSol::tsync();
        if (tl == 0) sm[WSol::SM_MISC + 1] = (double)atomicAdd(P.counter, 1);
        WSol::tsync();
        const int slot = (int)sm[WSol::SM_MISC + 1];
        if (slot >= P.B) {
            // convoy mode: keep answering the group's barriers until every warp of the CTA has run out of work
            if (P.convoy) while (wp::cta_count(false) != 0) {}
            break;
        }
        const int inst = P.order ? P.order[slot] : slot;   // longest-first scheduling when the caller has a predictor
        if ((unsigned)inst >= (unsigned)P.B) continue;      // not a permutation: never index outside the batch
        s.setup(inst);
        s.run();
    }
}

struct nmpc_handle {
    nmpc_desc d;
    nmpc_opts o;
    int ns, nc, M, S, n, mg, np, nnzj, nnzh, sm_count, dev;
    std::vector<int> jcol, jrow, hcol, hrow;  // CCS patterns (host)
    int *d_tables;
    NmpcEvalTables tb;
    long long launches;
    size_t ws_doubles_per_slot, solve_smem, eval_smem;
    int ctas_per_sm, lw, teams_per_cta, threads;
    const int *d_order;                       // optional processing order (device, caller owned), see nmpc_set_order
    int order_len;
    nmpc_tuning tune;
    int nobs, family, rk_steps;               // static obstacles per robot; family: 0 centralized, 1 obstacles, 2 small OCP (thread per instance)
    double *d_obs;                            // [nobs][3] on the device
    bool obs_in_p;                            // obstacle family with the geometry in p (per instance and stage): no d_obs
    bool tracking;                            // centralized family tracking a per-stage reference (nmpc_create_tracking)
    bool thread_ok;                           // a thread-per-instance kernel exists for this problem (small-OCP family; one robot with
                                              // static obstacles): used for the small-OCP family always, else from thread_min_batch on
    size_t t_ws_doubles;                      // its scratch per instance
    int thread_min_batch;
    int convoy;                               // warp path: iteration-level convoy of the CTA's warps (instruction-cache locality)
    bool block_path, eval_ok;                 // Nr > 10: CTA-per-instance dense-block solver; eval record fits shared memory
    int *d_pairs;                             // pair table (i, j) of the inequality rows, block path
    // host-pointer API staging
    char *d_buf;
    size_t d_bytes;
    cudaStream_t stream;
};

struct Trip { int r, c, tag; };

static void build_tables(nmpc_handle *h, std::vector<int> &tab)
{
    const int Nr = h->d.Nr, N = h->d.N, ns = h->ns, nc = h->nc, M = h->M, blk = ns + M, nX = ns * h->S;
    auto IX = [&](int k, int i, int c) { return k * ns + 3 * i + c; };
    auto IU = [&](int k, int i, int c) { return nX + k * nc + 2 * i + c; };
    std::vector<Trip> J, H;
    int tag = 0;
    // tags follow the layout of NmpcEvalTables: jac_rs | jac_ps | jac_init, then hes_rs | hes_ps
    for (int k = 0; k < N; k++)
        for (int i = 0; i < Nr; i++) {
            const int b = (k + 1) * blk, rx = b + 3 * i, ry = rx + 1, rt = rx + 2;
            const int rc[11][2] = {{rx, IX(k + 1, i, 0)}, {rx, IX(k, i, 0)}, {rx, IX(k, i, 2)}, {rx, IU(k, i, 0)},
                                   {ry, IX(k + 1, i, 1)}, {ry, IX(k, i, 1)}, {ry, IX(k, i, 2)}, {ry, IU(k, i, 0)},
                                   {rt, IX(k + 1, i, 2)}, {rt, IX(k, i, 2)}, {rt, IU(k, i, 1)}};
            for (auto &e : rc) J.push_back({e[0], e[1], tag++});
        }
    std::vector<std::pair<int, int>> pairs;
    for (int a = 0; a < Nr; a++)
        for (int b = a + 1; b < Nr; b++) pairs.push_back({a, b});
    for (int k = 0; k < N; k++)
        for (int q = 0; q < M; q++) {
            const int r = (k + 1) * blk + ns + q, i = pairs[q].first, j = pairs[q].second;
            J.push_back({r, IX(k, i, 0), tag++}); J.push_back({r, IX(k, j, 0), tag++});
            J.push_back({r, IX(k, i, 1), tag++}); J.push_back({r, IX(k, j, 1), tag++});
        }
    for (int r = 0; r < ns; r++) J.push_back({r, r, tag++});
    int htag = 0;
    for (int k = 0; k < N; k++)
        for (int i = 0; i < Nr; i++) {
            H.push_back({IX(k, i, 0), IX(k, i, 0), htag++}); H.push_back({IX(k, i, 1), IX(k, i, 1), htag++});
            H.push_back({IX(k, i, 2), IX(k, i, 2), htag++}); H.push_back({IU(k, i, 0), IX(k, i, 2), htag++});
            H.push_back({IU(k, i, 0), IU(k, i, 0), htag++}); H.push_back({IU(k, i, 1), IU(k, i, 1), htag++});
        }
    for (int k = 0; k < N; k++)
        for (int q = 0; q < M; q++) {
            H.push_back({IX(k, pairs[q].second, 0), IX(k, pairs[q].first, 0), htag++});
            H.push_back({IX(k, pairs[q].second, 1), IX(k, pairs[q].first, 1), htag++});
        }
    auto cmp = [](const Trip &a, const Trip &b) { return a.c != b.c ? a.c < b.c : a.r < b.r; };
    std::sort(J.begin(), J.end(), cmp);
    std::sort(H.begin(), H.end(), cmp);
    auto to_ccs = [&](const std::vector<Trip> &T, std::vector<int> &cp, std::vector<int> &ri, std::vector<int> &slot) {
        cp.assign(h->n + 1, 0); ri.resize(T.size()); slot.resize(T.size());
        for (size_t e = 0; e < T.size(); e++) { cp[T[e].c + 1]++; ri[e] = T[e].r; slot[T[e].tag] = (int)e; }
        for (int c = 0; c < h->n; c++) cp[c + 1] += cp[c];
    };
    std::vector<int> js, hs;
    to_ccs(J, h->jcol, h->jrow, js);
    to_ccs(H, h->hcol, h->hrow, hs);
    tab = js;
    tab.insert(tab.end(), hs.begin(), hs.end());
}

template <int NR, bool OBS = false, bool TRK = false> static size_t slot_doubles(int N) { return (size_t)WarpSolver<NR, OBS, TRK>::ws_doubles(N); }
template <int NR, bool OBS = false, bool TRK = false> static cudaError_t config_solve(nmpc_handle *h)
{
    typedef SolveCfg<NR, OBS, TRK> Cfg;
    h->lw = Cfg::LW; h->teams_per_cta = Cfg::TEAMS; h->threads = Cfg::THREADS;
    h->solve_smem = (size_t)Cfg::TEAMS * WarpSolver<NR, OBS, TRK>::SM_DOUBLES * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(solve_kernel<NR, OBS, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->solve_smem);
    if (e != cudaSuccess) return e;
    int nb = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, solve_kernel<NR, OBS, TRK>, Cfg::THREADS, h->solve_smem);
    h->ctas_per_sm = nb > 0 ? nb : 1;
    if (h->tune.ctas_per_sm >= 1 && h->tune.ctas_per_sm < h->ctas_per_sm) h->ctas_per_sm = h->tune.ctas_per_sm;
    return e;
}

static int create_impl(const nmpc_desc *d, const nmpc_opts *o, const nmpc_tuning *t, int nobs, const double *obs, bool obs_in_p,
                       bool tracking, nmpc_handle **out);

extern "C" void nmpc_default_tuning(nmpc_tuning *t)
{
    t->convoy = 2;   // measured: +14 % cold throughput over no convoy, +4 % over the iteration barrier alone
    t->ctas_per_sm = 0; t->force_block_path = 0; t->thread_min_batch = 0;
}

extern "C" int nmpc_create(const nmpc_desc *d, const nmpc_opts *o, nmpc_handle **out) { return create_impl(d, o, nullptr, 0, nullptr, false, false, out); }

static int check_obstacles(int n_obs, const double *obs)
{
    if (n_obs < 1 || n_obs > NMPC_MAX_OBSTACLES || !obs)
        return fail(NMPC_EINVAL, "nmpc_create_obstacles: need 1..%d obstacles (x, y, clearance radius each)", NMPC_MAX_OBSTACLES);
    for (int i = 0; i < n_obs; i++)
        if (!(obs[3 * i + 2] >= 0.0)) return fail(NMPC_EINVAL, "nmpc_create_obstacles: obstacle %d has a negative clearance radius", i);
    return 0;
}

extern "C" int nmpc_create_tuned(const nmpc_desc *d, const nmpc_opts *o, const nmpc_tuning *t, int n_obs, const double *obs, nmpc_handle **out)
{
    if (n_obs != 0) { int rc = check_obstacles(n_obs, obs); if (rc) return rc; }
    return create_impl(d, o, t, n_obs, n_obs ? obs : nullptr, false, false, out);
}

extern "C" int nmpc_create_obstacles(const nmpc_desc *d, const nmpc_opts *o, int n_obs, const double *obs, nmpc_handle **out)
{
    int rc = check_obstacles(n_obs, obs);
    if (rc) return rc;
    return create_impl(d, o, nullptr, n_obs, obs, false, false, out);
}

extern "C" int nmpc_create_moving_obstacles(const nmpc_desc *d, const nmpc_opts *o, const nmpc_tuning *t, int n_obs, nmpc_handle **out)
{
    if (n_obs < 1 || n_obs > NMPC_MAX_OBSTACLES)
        return fail(NMPC_EINVAL, "nmpc_create_moving_obstacles: need 1..%d obstacles, got %d", NMPC_MAX_OBSTACLES, n_obs);
    return create_impl(d, o, t, n_obs, nullptr, true, false, out);
}

extern "C" int nmpc_create_tracking(const nmpc_desc *d, const nmpc_opts *o, const nmpc_tuning *t, nmpc_handle **out)
{
    return create_impl(d, o, t, 0, nullptr, false, true, out);
}

// Small generic OCP family (thread per instance): currently the Van der Pol demo of mpc_pose_control_casadi.py
extern "C" int nmpc_create_ocp(int model, int N, double T, int rk_steps, const nmpc_opts *o, nmpc_handle **out)
{
    if (!out) return fail(NMPC_EINVAL, "nmpc_create_ocp: NULL argument");
    if (model != NMPC_OCP_VAN_DER_POL) return fail(NMPC_ENOTSUP, "nmpc_create_ocp: unknown model %d", model);
    if (N < 1 || !(T > 0) || rk_steps < 1) return fail(NMPC_EINVAL, "nmpc_create_ocp: need N >= 1, T > 0, rk_steps >= 1");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(NMPC_ECUDA, "nmpc_create_ocp: no CUDA device -- this library has no CPU fallback");
    nmpc_handle *h = new nmpc_handle();
    memset(&h->d, 0, sizeof h->d);
    h->d.Nr = 0; h->d.N = N; h->d.T = T;
    if (o) h->o = *o; else { nmpc_default_opts(&h->o); h->o.max_iter = 3000; }   // IPOPT's default max_iter: the demo sets no options
    typedef ThreadSolver<VanDerPol> TS;
    h->ns = TS::NX; h->nc = TS::NU; h->M = 0; h->S = N + 1; h->nobs = 0; h->family = 2; h->rk_steps = rk_steps;
    h->n = TS::NZ * N + TS::NX; h->mg = TS::NX * N; h->np = 0; h->nnzj = 0; h->nnzh = 0;
    h->launches = 0; h->d_buf = nullptr; h->d_bytes = 0; h->stream = nullptr; h->d_tables = nullptr; h->d_pairs = nullptr;
    h->d_order = nullptr; h->order_len = 0; h->d_obs = nullptr; h->block_path = false; h->eval_ok = false; h->thread_ok = true; h->thread_min_batch = 1;
    nmpc_default_tuning(&h->tune);
    cudaGetDevice(&h->dev);
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, h->dev);
    h->ws_doubles_per_slot = 0; h->t_ws_doubles = (size_t)TS::ws_doubles(N);
    h->lw = 0; h->teams_per_cta = 1; h->threads = 64; h->ctas_per_sm = 1; h->solve_smem = 0; h->eval_smem = 0;
    *out = h;
    return 0;
}

template <bool TRK> static cudaError_t eval_smem_attrs(int sz)
{
    cudaError_t e = cudaFuncSetAttribute(eval_kernel<0, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, sz);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(eval_kernel<1, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, sz);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(eval_kernel<2, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, sz);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(eval_kernel<3, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, sz);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(eval_kernel<4, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, sz);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(eval_kernel<5, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, sz);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(eval_kernel<6, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, sz);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(eval_kernel<7, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, sz);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(eval_kernel<8, TRK>, cudaFuncAttributeMaxDynamicSharedMemorySize, sz);
    return e;
}

static int create_impl(const nmpc_desc *d, const nmpc_opts *o, const nmpc_tuning *t, int nobs, const double *obs, bool obs_in_p,
                       bool tracking, nmpc_handle **out)
{
    if (!d || !out) return fail(NMPC_EINVAL, "nmpc_create: NULL argument");
    if (d->N < 1 || !(d->T > 0)) return fail(NMPC_EINVAL, "nmpc_create: need N >= 1 and T > 0");
    if (d->Nr < 1 || d->Nr > NMPC_MAX_ROBOTS)
        return fail(NMPC_ENOTSUP, "nmpc_create: Nr = %d; supported: 1..10 robots (warp-per-instance) and 11..%d (CTA-per-instance dense blocks)", d->Nr, NMPC_MAX_ROBOTS);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(NMPC_ECUDA, "nmpc_create: no CUDA device -- this library has no CPU fallback");
    nmpc_handle *h = new nmpc_handle();
    h->d = *d;
    if (o) h->o = *o; else nmpc_default_opts(&h->o);
    if (t) h->tune = *t; else nmpc_default_tuning(&h->tune);
    h->ns = 3 * d->Nr; h->nc = 2 * d->Nr; h->M = d->Nr * (d->Nr - 1) / 2; h->S = d->N + 1;
    h->nobs = nobs; h->family = nobs > 0 ? 1 : 0; h->d_obs = nullptr; h->obs_in_p = obs_in_p; h->tracking = tracking;
    // p = [x0bar; xs], then with the obstacles in p one [nobs][3] table per stage k = 0..N-1; tracking: p = [x0bar; Z[N][5 Nr]]
    h->n = h->ns * h->S + h->nc * d->N;
    h->np = tracking ? h->ns + d->N * (h->ns + h->nc) : 2 * h->ns + (obs_in_p ? 3 * d->N * nobs : 0);
    // row layout: family 0 = (N+1) blocks of [ns equality rows ; M pair rows]; family 1 (static obstacles) = ns rows, then N
    // blocks of [ns ; M + Nr n_obs]   (first_scenario_mpc_obstacle_avoidance.py:109-125)
    h->mg = h->family ? h->ns + d->N * (h->ns + h->M + d->Nr * nobs) : h->S * (h->ns + h->M);
    h->nnzj = 3 * d->Nr + d->N * (11 * d->Nr + 4 * h->M); h->nnzh = d->N * (6 * d->Nr + 2 * h->M);
    h->launches = 0; h->d_buf = nullptr; h->d_bytes = 0; h->stream = nullptr; h->d_tables = nullptr;
    h->d_pairs = nullptr; h->d_order = nullptr; h->order_len = 0;
    // the obstacle family runs on the dense-block path for every Nr; nmpc_tuning.force_block_path: test hook, any Nr on that path
    // the obstacle family runs on the warp-per-instance path for up to 4 robots while its rows fit the warp's lanes (pair rows +
    // Nr n_obs <= 32: one robot with up to 32 obstacles; the reference's scripts have one robot and 1, 4 or 6), else on the dense-block path
    const int lanes = 32;
    const bool obs_fit = d->Nr <= NMPC_OBS_WARP_MAX_ROBOTS && h->M + d->Nr * nobs <= lanes;
    h->block_path = d->Nr > 10 || (h->family != 0 && !obs_fit) || h->tune.force_block_path != 0; h->eval_ok = h->family == 0;
    // A single robot with static obstacles (the reference's obstacle scripts) also runs on the thread-per-instance small-OCP
    // solver (UnicycleObstacles model), parity-tested, but measured slower than the CTA-per-instance path both alone (88 ms
    // against 49 ms per solve at N = 100) and in batches (9.2 k against 23.0 k solves/s, B = 8192, N = 20: its per-thread
    // scratch is not coalesced across instances), so it is off unless nmpc_tuning.thread_min_batch sets a switch-over batch size.
    // (the thread-per-instance solver takes one static table: never for obstacles in p)
    h->thread_ok = h->family == 1 && d->Nr == 1 && !obs_in_p;
    h->t_ws_doubles = h->thread_ok ? (size_t)ThreadSolver<UnicycleObstacles>::ws_doubles(d->N) : 0;
    h->thread_min_batch = h->tune.thread_min_batch > 0 ? h->tune.thread_min_batch : 0x7fffffff;
    h->convoy = h->tune.convoy;   // 0 off, 1 barrier per iteration, 2 also before the forward pass
    cudaGetDevice(&h->dev);
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, h->dev);
    std::vector<int> tab;
    build_tables(h, tab);
    cudaError_t e = cudaMalloc(&h->d_tables, tab.size() * sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_tables, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { nmpc_destroy(h); return fail(NMPC_ECUDA, "nmpc_create: table upload failed: %s", cudaGetErrorString(e)); }
    const int N = d->N, Nr = d->Nr, M = h->M;
    h->tb.jac_rs = h->d_tables;
    h->tb.jac_ps = h->tb.jac_rs + (size_t)N * Nr * 11;
    h->tb.jac_init = h->tb.jac_ps + (size_t)N * M * 4;
    h->tb.hes_rs = h->d_tables + h->nnzj;
    h->tb.hes_ps = h->tb.hes_rs + (size_t)N * Nr * 6;
    switch (h->block_path ? 0 : (h->family ? 100 + Nr : (tracking ? 200 + Nr : Nr))) {
#ifndef NMPC_DEV_ONLY_NR
        case 201: h->ws_doubles_per_slot = slot_doubles<1, false, true>(N); e = config_solve<1, false, true>(h); break;
        case 202: h->ws_doubles_per_slot = slot_doubles<2, false, true>(N); e = config_solve<2, false, true>(h); break;
        case 203: h->ws_doubles_per_slot = slot_doubles<3, false, true>(N); e = config_solve<3, false, true>(h); break;
        case 204: h->ws_doubles_per_slot = slot_doubles<4, false, true>(N); e = config_solve<4, false, true>(h); break;
        case 205: h->ws_doubles_per_slot = slot_doubles<5, false, true>(N); e = config_solve<5, false, true>(h); break;
        case 206: h->ws_doubles_per_slot = slot_doubles<6, false, true>(N); e = config_solve<6, false, true>(h); break;
        case 207: h->ws_doubles_per_slot = slot_doubles<7, false, true>(N); e = config_solve<7, false, true>(h); break;
        case 208: h->ws_doubles_per_slot = slot_doubles<8, false, true>(N); e = config_solve<8, false, true>(h); break;
        case 209: h->ws_doubles_per_slot = slot_doubles<9, false, true>(N); e = config_solve<9, false, true>(h); break;
        case 210: h->ws_doubles_per_slot = slot_doubles<10, false, true>(N); e = config_solve<10, false, true>(h); break;
        case 101: h->ws_doubles_per_slot = slot_doubles<1, true>(N); e = config_solve<1, true>(h); break;
        case 102: h->ws_doubles_per_slot = slot_doubles<2, true>(N); e = config_solve<2, true>(h); break;
        case 103: h->ws_doubles_per_slot = slot_doubles<3, true>(N); e = config_solve<3, true>(h); break;
        case 104: h->ws_doubles_per_slot = slot_doubles<4, true>(N); e = config_solve<4, true>(h); break;
#endif
#ifdef NMPC_DEV_ONLY_NR   // development builds (tools/dev_build.sh): one warp-path instantiation, 5 x faster to compile
        case NMPC_DEV_ONLY_NR: h->ws_doubles_per_slot = slot_doubles<NMPC_DEV_ONLY_NR>(N); e = config_solve<NMPC_DEV_ONLY_NR>(h); break;
        case 1000: break;
#define NMPC_SKIP_OTHER_NR
#endif
#ifndef NMPC_SKIP_OTHER_NR
        case 1: h->ws_doubles_per_slot = slot_doubles<1>(N); e = config_solve<1>(h); break;
        case 2: h->ws_doubles_per_slot = slot_doubles<2>(N); e = config_solve<2>(h); break;
        case 3: h->ws_doubles_per_slot = slot_doubles<3>(N); e = config_solve<3>(h); break;
        case 4: h->ws_doubles_per_slot = slot_doubles<4>(N); e = config_solve<4>(h); break;
        case 5: h->ws_doubles_per_slot = slot_doubles<5>(N); e = config_solve<5>(h); break;
        case 6: h->ws_doubles_per_slot = slot_doubles<6>(N); e = config_solve<6>(h); break;
        case 7: h->ws_doubles_per_slot = slot_doubles<7>(N); e = config_solve<7>(h); break;
        case 8: h->ws_doubles_per_slot = slot_doubles<8>(N); e = config_solve<8>(h); break;
        case 9: h->ws_doubles_per_slot = slot_doubles<9>(N); e = config_solve<9>(h); break;
        case 10: h->ws_doubles_per_slot = slot_doubles<10>(N); e = config_solve<10>(h); break;
#endif
        default: {   // dense-block path: one 512-thread CTA per instance, the control block of the stage matrix in shared memory
            h->ws_doubles_per_slot = (size_t)BlockSolver::ws_doubles(Nr, N, h->nobs);
            // CTA size: the register-resident Cholesky needs 8 rows per warp over ncp = roundup(2 Nr, 32) rows, i.e. 4 ncp threads
            // (128 for 11..16 robots, 512 for 49..64); smaller swarms then fit several CTAs per SM
            h->lw = BlockSolver::row_width(Nr, h->nobs); h->teams_per_cta = 1;
            h->threads = 4 * ((2 * Nr + 31) & ~31);
            if (h->threads > NMPC_BLOCK_THREADS) h->threads = NMPC_BLOCK_THREADS;
            h->solve_smem = (size_t)BlockSolver::sm_doubles(Nr) * sizeof(double);
            e = cudaFuncSetAttribute(solve_kernel_block, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->solve_smem);
            int nb = 0;
            if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, solve_kernel_block, h->threads, h->solve_smem);
            h->ctas_per_sm = nb > 0 ? nb : 1;
            if (h->tune.ctas_per_sm >= 1 && h->tune.ctas_per_sm < h->ctas_per_sm) h->ctas_per_sm = h->tune.ctas_per_sm;
            std::vector<int> pr;
            for (int a = 0; a < Nr; a++)
                for (int b = a + 1; b < Nr; b++) { pr.push_back(a); pr.push_back(b); }
            if (e == cudaSuccess) e = cudaMalloc(&h->d_pairs, (pr.size() + 2) * sizeof(int));
            if (e == cudaSuccess && !pr.empty()) e = cudaMemcpy(h->d_pairs, pr.data(), pr.size() * sizeof(int), cudaMemcpyHostToDevice);
            break;
        }
    }
    if (e == cudaSuccess && h->nobs > 0 && !obs_in_p) {
        e = cudaMalloc(&h->d_obs, (size_t)3 * h->nobs * sizeof(double));
        if (e == cudaSuccess) e = cudaMemcpy(h->d_obs, obs, (size_t)3 * h->nobs * sizeof(double), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) { nmpc_destroy(h); return fail(NMPC_ECUDA, "nmpc_create: kernel configuration failed: %s", cudaGetErrorString(e)); }
    // the record stages all of p: 2 ns values, or a tracking handle's ns + N nz
    h->eval_smem = (size_t)(2 * h->n + 2 * h->mg + h->np + h->nnzj + h->nnzh + 32 + 8) * sizeof(double);
    if (h->eval_smem > (size_t)220 * 1024 || h->family != 0) h->eval_ok = false;   // large swarms: the stand-alone evaluation record exceeds shared memory
    else e = tracking ? eval_smem_attrs<true>((int)h->eval_smem) : eval_smem_attrs<false>((int)h->eval_smem);
    if (e != cudaSuccess) { const size_t es = h->eval_smem; nmpc_destroy(h); return fail(NMPC_ENOTSUP, "nmpc_create: eval record (%zu B) exceeds shared memory: %s", es, cudaGetErrorString(e)); }
    *out = h;
    return 0;
}

extern "C" void nmpc_destroy(nmpc_handle *h)
{
    if (!h) return;
    if (h->d_tables) cudaFree(h->d_tables);
    if (h->d_pairs) cudaFree(h->d_pairs);
    if (h->d_obs) cudaFree(h->d_obs);
    if (h->d_buf) cudaFree(h->d_buf);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

extern "C" int nmpc_n(const nmpc_handle *h) { return h ? h->n : NMPC_EINVAL; }
extern "C" int nmpc_mg(const nmpc_handle *h) { return h ? h->mg : NMPC_EINVAL; }
extern "C" int nmpc_np(const nmpc_handle *h) { return h ? h->np : NMPC_EINVAL; }
extern "C" int nmpc_nnz_jac(const nmpc_handle *h) { return h ? h->nnzj : NMPC_EINVAL; }
extern "C" int nmpc_nnz_hess(const nmpc_handle *h) { return h ? h->nnzh : NMPC_EINVAL; }
extern "C" long long nmpc_launch_count(const nmpc_handle *h) { return h ? h->launches : 0; }

extern "C" int nmpc_jac_pattern(const nmpc_handle *h, int32_t *colptr, int32_t *rowidx)
{
    if (!h || !colptr || !rowidx) return fail(NMPC_EINVAL, "nmpc_jac_pattern: NULL argument");
    if (h->family) return fail(NMPC_ENOTSUP, "nmpc_jac_pattern: not available for the static-obstacle family");
    memcpy(colptr, h->jcol.data(), sizeof(int) * (h->n + 1)); memcpy(rowidx, h->jrow.data(), sizeof(int) * h->nnzj);
    return 0;
}
extern "C" int nmpc_hess_pattern(const nmpc_handle *h, int32_t *colptr, int32_t *rowidx)
{
    if (!h || !colptr || !rowidx) return fail(NMPC_EINVAL, "nmpc_hess_pattern: NULL argument");
    if (h->family) return fail(NMPC_ENOTSUP, "nmpc_hess_pattern: not available for the static-obstacle family");
    memcpy(colptr, h->hcol.data(), sizeof(int) * (h->n + 1)); memcpy(rowidx, h->hrow.data(), sizeof(int) * h->nnzh);
    return 0;
}

static int solve_grid(const nmpc_handle *h, int B)
{
    int need = (B + h->teams_per_cta - 1) / h->teams_per_cta, cap = h->sm_count * h->ctas_per_sm;
    return need < cap ? (need > 0 ? need : 1) : cap;
}
static size_t bound_rows_bytes(const nmpc_handle *h, int nb) { return (size_t)nb * NMPC_BR_COUNT * h->S * h->lw * sizeof(double); }
static bool use_thread(const nmpc_handle *h, int B) { return h->thread_ok && B >= h->thread_min_batch; }
static size_t ws_bytes_for(const nmpc_handle *h, int B, int nb)
{
    if (use_thread(h, B)) return 256 + (size_t)((B + 63) / 64 * 64) * h->t_ws_doubles * sizeof(double);
    return 256 + bound_rows_bytes(h, nb) + (size_t)solve_grid(h, B) * h->teams_per_cta * h->ws_doubles_per_slot * sizeof(double);
}
extern "C" size_t nmpc_workspace_bytes(const nmpc_handle *h, int B) { return h && B > 0 ? ws_bytes_for(h, B, 1) : 0; }
extern "C" size_t nmpc_workspace_bytes_batched_bounds(const nmpc_handle *h, int B) { return h && B > 0 ? ws_bytes_for(h, B, B) : 0; }

static int solve_impl(nmpc_handle *h, int B, const double *x0, const double *p, const double *lbx, const double *ubx,
                      const double *lbg, const double *ubg, int bounds_batched, double *x, double *f, double *g,
                      double *lam_x, double *lam_g, int32_t *status, int32_t *iters, double *stats, double *trace,
                      int max_trace, void *workspace, size_t workspace_bytes, cudaStream_t st)
{
    if (!h || !x0 || (!p && h->np > 0) || !lbx || !ubx || !lbg || !ubg || !x || !workspace) return fail(NMPC_EINVAL, "nmpc_solve: NULL argument");
    if (B <= 0) return fail(NMPC_EINVAL, "nmpc_solve: B must be positive");
    if (h->d_order && h->order_len != B)
        return fail(NMPC_EINVAL, "nmpc_solve: the scheduling order set with nmpc_set_order has %d entries, the batch has %d", h->order_len, B);
    {
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess || cur != h->dev)
            return fail(NMPC_EINVAL, "nmpc_solve: the handle was created on CUDA device %d but device %d is current", h->dev, cur);
    }
    const int nb = bounds_batched ? B : 1;
    const size_t need = ws_bytes_for(h, B, nb);
    if (workspace_bytes < need) return fail(NMPC_ENOMEM, "nmpc_solve: workspace %zu B < %zu B required", workspace_bytes, need);
    const bool thr = use_thread(h, B);
    char *base = (char *)workspace;
    int *counter = (int *)base, *berr = counter + 1;
    double *brows = (double *)(base + 256);
    double *slots = (double *)(base + 256 + (thr ? 0 : bound_rows_bytes(h, nb)));
    CUDA_OK(cudaMemsetAsync(base, 0, 256, st));
    if (!thr) {
        long long total = (long long)nb * h->S * h->lw;
        int blocks = (int)std::min<long long>((total + 255) / 256, 4096);
        prep_bounds_kernel<<<blocks, 256, 0, st>>>(h->d.Nr, h->d.N, h->o.bound_relax_factor, nb, h->lw, lbx, ubx, lbg, ubg, brows, berr, h->nobs, h->family, h->block_path ? 0 : 1);
        h->launches++;
    }
    NmpcSolveParams P;
    memset(&P, 0, sizeof P);
    P.Nr = h->d.Nr; P.N = h->d.N; P.B = B; P.T = h->d.T;
    memcpy(P.Q, h->d.Q, sizeof P.Q); memcpy(P.R, h->d.R, sizeof P.R);
    P.o = h->o; P.x0 = x0; P.p = p; P.brows = brows;
    P.bstride = bounds_batched ? (long long)NMPC_BR_COUNT * h->S * h->lw : 0;
    P.bound_err = berr; P.x = x; P.f = f; P.g = g; P.lam_x = lam_x; P.lam_g = lam_g; P.status = status; P.iters = iters;
    P.stats = stats; P.trace = trace; P.max_trace = max_trace; P.ws = slots; P.ws_stride = (long long)(thr ? h->t_ws_doubles : h->ws_doubles_per_slot);
    P.counter = counter; P.pairs = h->d_pairs; P.order = h->d_order; P.nobs = h->nobs; P.family = h->family; P.obs = h->d_obs;
    // convoy: one-warp teams only (measured -5..-8 % for the two-warp teams of 7..10 robots, whose groups are two instances),
    // and pointless while every CTA has at most one working team
    P.convoy = (!h->block_path && !thr && h->lw == 32 && h->teams_per_cta > 1 && B > solve_grid(h, B)) ? h->convoy : 0;
    P.lbx = lbx; P.ubx = ubx; P.lbg = lbg; P.ubg = ubg; P.bounds_batched = bounds_batched; P.rk_steps = h->rk_steps; P.np = h->np; P.obs_in_p = h->obs_in_p;
    const int grid = thr ? (B + 63) / 64 : solve_grid(h, B);
    if (thr && h->family == 2) solve_kernel_small_ocp<VanDerPol><<<grid, 64, 0, st>>>(P);
    else if (thr) solve_kernel_small_ocp<UnicycleObstacles><<<grid, 64, 0, st>>>(P);
    else if (h->block_path) solve_kernel_block<<<grid, h->threads, h->solve_smem, st>>>(P);
    else switch (h->family ? 100 + h->d.Nr : (h->tracking ? 200 + h->d.Nr : h->d.Nr)) {
#ifndef NMPC_DEV_ONLY_NR
        case 201: solve_kernel<1, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 202: solve_kernel<2, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 203: solve_kernel<3, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 204: solve_kernel<4, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 205: solve_kernel<5, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 206: solve_kernel<6, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 207: solve_kernel<7, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 208: solve_kernel<8, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 209: solve_kernel<9, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 210: solve_kernel<10, false, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 101: solve_kernel<1, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 102: solve_kernel<2, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 103: solve_kernel<3, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 104: solve_kernel<4, true><<<grid, h->threads, h->solve_smem, st>>>(P); break;
#endif
#ifdef NMPC_DEV_ONLY_NR
        default: solve_kernel<NMPC_DEV_ONLY_NR><<<grid, h->threads, h->solve_smem, st>>>(P); break;
#else
        case 1: solve_kernel<1><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 2: solve_kernel<2><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 3: solve_kernel<3><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 4: solve_kernel<4><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 5: solve_kernel<5><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 6: solve_kernel<6><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 7: solve_kernel<7><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 8: solve_kernel<8><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        case 9: solve_kernel<9><<<grid, h->threads, h->solve_smem, st>>>(P); break;
        default: solve_kernel<10><<<grid, h->threads, h->solve_smem, st>>>(P); break;
#endif
    }
    h->launches++;
    CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int nmpc_set_order(nmpc_handle *h, const int32_t *order, int len)
{
    if (!h) return fail(NMPC_EINVAL, "nmpc_set_order: NULL handle");
    if (order && len <= 0) return fail(NMPC_EINVAL, "nmpc_set_order: len must be positive");
    h->d_order = order; h->order_len = order ? len : 0;
    return 0;
}

extern "C" int nmpc_solve(nmpc_handle *h, int B, const double *x0, const double *p, const double *lbx, const double *ubx,
                          const double *lbg, const double *ubg, int bounds_batched, double *x, double *f, double *g,
                          double *lam_x, double *lam_g, int32_t *status, int32_t *iters, double *stats, void *workspace,
                          size_t workspace_bytes, void *stream)
{
    return solve_impl(h, B, x0, p, lbx, ubx, lbg, ubg, bounds_batched, x, f, g, lam_x, lam_g, status, iters, stats, nullptr, 0,
                      workspace, workspace_bytes, (cudaStream_t)stream);
}

// debugging / parity entry: same as nmpc_solve plus a per-iteration trace [B][max_trace][8]
extern "C" int nmpc_solve_trace(nmpc_handle *h, int B, const double *x0, const double *p, const double *lbx, const double *ubx,
                                const double *lbg, const double *ubg, int bounds_batched, double *x, double *f, double *g,
                                double *lam_x, double *lam_g, int32_t *status, int32_t *iters, double *stats, double *trace,
                                int max_trace, void *workspace, size_t workspace_bytes, void *stream)
{
    return solve_impl(h, B, x0, p, lbx, ubx, lbg, ubg, bounds_batched, x, f, g, lam_x, lam_g, status, iters, stats, trace, max_trace,
                      workspace, workspace_bytes, (cudaStream_t)stream);
}

static size_t al(size_t v) { return (v + 255) & ~(size_t)255; }

extern "C" int nmpc_solve_host(nmpc_handle *h, int B, const double *x0, const double *p, const double *lbx, const double *ubx,
                               const double *lbg, const double *ubg, int bounds_batched, double *x, double *f, double *g,
                               double *lam_x, double *lam_g, int32_t *status, int32_t *iters, double *stats)
{
    if (!h || !x0 || (!p && h->np > 0) || !lbx || !ubx || !lbg || !ubg || !x) return fail(NMPC_EINVAL, "nmpc_solve_host: NULL argument");
    if (B <= 0) return fail(NMPC_EINVAL, "nmpc_solve_host: B must be positive");
    const int nb = bounds_batched ? B : 1;
    const size_t n = h->n, mg = h->mg, np = h->np, D = sizeof(double);
    const size_t o_x0 = 0, o_p = o_x0 + al(B * n * D), o_lbx = o_p + al(B * np * D), o_ubx = o_lbx + al(nb * n * D),
                 o_lbg = o_ubx + al(nb * n * D), o_ubg = o_lbg + al(nb * mg * D), o_x = o_ubg + al(nb * mg * D),
                 o_f = o_x + al(B * n * D), o_g = o_f + al(B * D), o_lx = o_g + al(B * mg * D), o_lg = o_lx + al(B * n * D),
                 o_st = o_lg + al(B * mg * D), o_it = o_st + al(B * 4), o_stats = o_it + al(B * 4),
                 o_ws = o_stats + al((size_t)B * NMPC_NSTATS * D);
    const size_t wsb = ws_bytes_for(h, B, nb), total = o_ws + wsb;
    if (!h->stream) CUDA_OK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    if (h->d_bytes < total) {
        if (h->d_buf) cudaFree(h->d_buf);
        h->d_buf = nullptr; h->d_bytes = 0;
        CUDA_OK(cudaMalloc(&h->d_buf, total));
        h->d_bytes = total;
    }
    char *b = h->d_buf;
    cudaStream_t st = h->stream;
    CUDA_OK(cudaMemcpyAsync(b + o_x0, x0, B * n * D, cudaMemcpyHostToDevice, st));
    if (np > 0) CUDA_OK(cudaMemcpyAsync(b + o_p, p, B * np * D, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemcpyAsync(b + o_lbx, lbx, nb * n * D, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemcpyAsync(b + o_ubx, ubx, nb * n * D, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemcpyAsync(b + o_lbg, lbg, nb * mg * D, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemcpyAsync(b + o_ubg, ubg, nb * mg * D, cudaMemcpyHostToDevice, st));
    int rc = solve_impl(h, B, (double *)(b + o_x0), (double *)(b + o_p), (double *)(b + o_lbx), (double *)(b + o_ubx),
                        (double *)(b + o_lbg), (double *)(b + o_ubg), bounds_batched, (double *)(b + o_x),
                        f ? (double *)(b + o_f) : nullptr, g ? (double *)(b + o_g) : nullptr,
                        lam_x ? (double *)(b + o_lx) : nullptr, lam_g ? (double *)(b + o_lg) : nullptr, (int32_t *)(b + o_st),
                        iters ? (int32_t *)(b + o_it) : nullptr, stats ? (double *)(b + o_stats) : nullptr, nullptr, 0, b + o_ws,
                        wsb, st);
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(x, b + o_x, B * n * D, cudaMemcpyDeviceToHost, st));
    if (f) CUDA_OK(cudaMemcpyAsync(f, b + o_f, B * D, cudaMemcpyDeviceToHost, st));
    if (g) CUDA_OK(cudaMemcpyAsync(g, b + o_g, B * mg * D, cudaMemcpyDeviceToHost, st));
    if (lam_x) CUDA_OK(cudaMemcpyAsync(lam_x, b + o_lx, B * n * D, cudaMemcpyDeviceToHost, st));
    if (lam_g) CUDA_OK(cudaMemcpyAsync(lam_g, b + o_lg, B * mg * D, cudaMemcpyDeviceToHost, st));
    std::vector<int32_t> st_host;
    int32_t *stp = status;
    if (!stp) { st_host.resize(B); stp = st_host.data(); }
    CUDA_OK(cudaMemcpyAsync(stp, b + o_st, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    if (iters) CUDA_OK(cudaMemcpyAsync(iters, b + o_it, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    if (stats) CUDA_OK(cudaMemcpyAsync(stats, b + o_stats, (size_t)B * NMPC_NSTATS * D, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    // the warp and block paths reject the whole batch, the thread path only the instance whose bounds are bad: look at all
    for (int i = 0; i < B; i++)
        if (stp[i] < 0)
            return fail(stp[i], "nmpc_solve_host: bounds of instance %d rejected (%s)", i,
                        stp[i] == NMPC_EBOUNDS ? "lb > ub" : "fixed variable, non-equality dynamics row or equality distance row");
    return 0;
}

extern "C" int nmpc_shift(nmpc_handle *h, int B, const double *x_prev, double *x0_next, void *stream)
{
    if (!h || !x_prev || !x0_next || B <= 0) return fail(NMPC_EINVAL, "nmpc_shift: bad argument");
    if (h->family == 2) return fail(NMPC_ENOTSUP, "nmpc_shift: the small-OCP family is a single solve, it has no MPC shift");
    if (x_prev == x0_next) return fail(NMPC_EINVAL, "nmpc_shift: in-place shift is not supported");
    long long total = (long long)B * h->n;
    int blocks = (int)std::min<long long>(B, (long long)h->sm_count * 8);
    shift_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(h->d.Nr, h->d.N, total, x_prev, x0_next);
    h->launches++;
    CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int nmpc_plant(nmpc_handle *h, int B, const double *state, const double *x_opt, double *state_next, void *stream)
{
    if (!h || !state || !x_opt || !state_next || B <= 0) return fail(NMPC_EINVAL, "nmpc_plant: bad argument");
    if (h->family == 2) return fail(NMPC_ENOTSUP, "nmpc_plant: not available for the small-OCP family");
    int blocks = std::min((B * h->d.Nr + 255) / 256, h->sm_count * 16);
    plant_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(h->d.Nr, h->d.N, h->d.T, B, state, x_opt, state_next);
    h->launches++;
    CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int nmpc_eval(nmpc_handle *h, int B, const double *w, const double *p, const double *lam_g, double *f, double *grad,
                         double *g, double *jac, double *hess, void *stream)
{
    if (!h || !w || !p || B <= 0) return fail(NMPC_EINVAL, "nmpc_eval: bad argument");
    if (hess && !lam_g) return fail(NMPC_EINVAL, "nmpc_eval: hess needs lam_g");
    if (h->family) return fail(NMPC_ENOTSUP, "nmpc_eval: not available for this problem family");
    if (!h->eval_ok) {   // record larger than shared memory: global-memory variant
        eval_kernel_big<<<std::min(B, h->sm_count * 8), 256, 0, (cudaStream_t)stream>>>(h->d.Nr, h->d.N, h->d.T, h->d.Q[0], h->d.Q[1], h->d.Q[2],
                                                                                        h->d.R[0], h->d.R[1], B, w, p, lam_g, f, grad, g, jac, hess, h->tb,
                                                                                        h->np, h->tracking ? h->ns + h->nc : 0);
        h->launches++;
        CUDA_OK(cudaGetLastError());
        return 0;
    }
    int per_sm = (int)std::max<size_t>(1, (size_t)(220 * 1024) / h->eval_smem);
    int blocks = std::min(B, h->sm_count * per_sm);
    const int pf = (std::max(h->n, h->mg) + 255) / 256;
#define EVAL_LAUNCH(PFV)                                                                                                          \
    do {                                                                                                                          \
        if (h->tracking)                                                                                                          \
            eval_kernel<PFV, true><<<blocks, 256, h->eval_smem, (cudaStream_t)stream>>>(h->d.Nr, h->d.N, h->d.T, h->d.Q[0], h->d.Q[1], \
                h->d.Q[2], h->d.R[0], h->d.R[1], B, w, p, lam_g, f, grad, g, jac, hess, h->tb);                                    \
        else                                                                                                                      \
            eval_kernel<PFV, false><<<blocks, 256, h->eval_smem, (cudaStream_t)stream>>>(h->d.Nr, h->d.N, h->d.T, h->d.Q[0], h->d.Q[1], \
                h->d.Q[2], h->d.R[0], h->d.R[1], B, w, p, lam_g, f, grad, g, jac, hess, h->tb);                                    \
    } while (0)
    switch (pf <= 8 ? pf : 0) {
        case 1: EVAL_LAUNCH(1); break; case 2: EVAL_LAUNCH(2); break; case 3: EVAL_LAUNCH(3); break; case 4: EVAL_LAUNCH(4); break;
        case 5: EVAL_LAUNCH(5); break; case 6: EVAL_LAUNCH(6); break; case 7: EVAL_LAUNCH(7); break; case 8: EVAL_LAUNCH(8); break;
        default: EVAL_LAUNCH(0); break;
    }
#undef EVAL_LAUNCH
    h->launches++;
    CUDA_OK(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------
// FP64 FMA-pipe probe: the roofline denominator for the factorisation (MEASURED_PEAKS.json holds
// only HBM and bf16 figures).  8 independent DFMA chains per thread, 148 x 8 CTAs of 256 threads.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_probe_kernel(int iters, double *out)
{
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; i++) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    double r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (r == 123.456) out[0] = r;
}

// FP64 tensor-core probe: mma.sync.aligned.m8n8k4 f64 (DMMA), 8 independent accumulator tiles per warp, register only.
// One instruction = 8 x 8 x 4 FMAs = 512 flop per warp.  Measured beside the DFMA probe: on B200 the two have the same peak and share one pipe
// (tools/probe_fp64_mix.cu), so DMMA does not raise the FP64 roofline; the dense-block path (block_solver.cuh) uses it for its
// contractions because it needs a quarter of the operand traffic of 4 x 4 register tiles.
__global__ void __launch_bounds__(256) dmma_probe_kernel(int iters, double *out)
{
    double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
    double c[8][2];
    for (int t = 0; t < 8; t++) { c[t][0] = t * 1e-3; c[t][1] = t * 2e-3; }
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int t = 0; t < 8; t++)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                         : "+d"(c[t][0]), "+d"(c[t][1]) : "d"(a), "d"(b));
    }
    double r = 0.0;
    for (int t = 0; t < 8; t++) r += c[t][0] + c[t][1];
    if (r == 123.456) out[0] = r;
}

// debug aid: cycle counters per phase of the dense-block factorisation (CTA 0); reset = 1 clears them after the read
extern "C" int nmpc_debug_block_profile(long long *out16, int reset)
{
    if (!out16) return fail(NMPC_EINVAL, "nmpc_debug_block_profile: NULL argument");
    CUDA_OK(cudaMemcpyFromSymbol(out16, g_block_prof, sizeof(long long) * 16));
    if (reset) { long long z[16] = {0}; CUDA_OK(cudaMemcpyToSymbol(g_block_prof, z, sizeof z)); }
    return 0;
}

extern "C" int nmpc_probe_fp64(double *tflops_out)
{
    if (!tflops_out) return fail(NMPC_EINVAL, "nmpc_probe_fp64: NULL argument");
    int dev = 0, sms = 0;
    CUDA_OK(cudaGetDevice(&dev));
    CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    double *d = nullptr;
    CUDA_OK(cudaMalloc(&d, 64));
    cudaEvent_t e0, e1;
    CUDA_OK(cudaEventCreate(&e0)); CUDA_OK(cudaEventCreate(&e1));
    const int iters = 1 << 16, grid = sms * 8;
    double best = 0.0;
    for (int rep = 0; rep < 5; rep++) {
        CUDA_OK(cudaEventRecord(e0));
        dfma_probe_kernel<<<grid, 256>>>(iters, d);
        CUDA_OK(cudaEventRecord(e1));
        CUDA_OK(cudaEventSynchronize(e1));
        float ms = 0;
        CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
        double tf = 2.0 * 8.0 * iters * 256.0 * grid / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    *tflops_out = best;
    return 0;
}

extern "C" int nmpc_probe_dmma(double *tflops_out)
{
    if (!tflops_out) return fail(NMPC_EINVAL, "nmpc_probe_dmma: NULL argument");
    int dev = 0, sms = 0;
    CUDA_OK(cudaGetDevice(&dev));
    CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    double *d = nullptr;
    CUDA_OK(cudaMalloc(&d, 64));
    cudaEvent_t e0, e1;
    CUDA_OK(cudaEventCreate(&e0)); CUDA_OK(cudaEventCreate(&e1));
    const int iters = 1 << 14, grid = sms * 8;
    double best = 0.0;
    for (int rep = 0; rep < 5; rep++) {
        CUDA_OK(cudaEventRecord(e0));
        dmma_probe_kernel<<<grid, 256>>>(iters, d);
        CUDA_OK(cudaEventRecord(e1));
        CUDA_OK(cudaEventSynchronize(e1));
        float ms = 0;
        CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
        double tf = 512.0 * 8.0 * iters * 8.0 * grid / (ms * 1e-3) / 1e12;   // 512 flop x 8 tiles x 8 warps per CTA
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    *tflops_out = best;
    return 0;
}
