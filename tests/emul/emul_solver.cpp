// CPU fibre emulation of the product's warp-per-instance solver -- TEST INFRASTRUCTURE ONLY.
// Compiles csrc/solver_body.cuh (unchanged) against tests/emul/warp_prims.cuh.  Never shipped,
// never on the product path: the product fails loudly without its CUDA library.
#include "warp_prims.cuh"
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "solver_body.cuh"
#include "bounds_prep.cuh"

namespace wp { thread_local Emu *emu = nullptr; }

namespace {
struct Job { const NmpcSolveParams *P; int inst; double *sm, *ws; int Nr; };
thread_local Job job;

template <int NR> void lane_body()
{
    if (NR <= 4 && job.P->nobs > 0) {   // the static-obstacle family has its own instantiation (1..4 robots on the warp path)
        WarpSolver<(NR <= 4 ? NR : 1), true> s(*job.P, job.sm, job.ws);
        s.init_team();
        s.setup(job.inst);
        s.run();
        return;
    }
    WarpSolver<NR> s(*job.P, job.sm, job.ws);
    s.init_team();
    s.setup(job.inst);
    s.run();
}
void fibre_main()
{
    switch (job.Nr) {
        case 1: lane_body<1>(); break; case 2: lane_body<2>(); break; case 3: lane_body<3>(); break;
        case 4: lane_body<4>(); break; case 5: lane_body<5>(); break; case 6: lane_body<6>(); break;
        case 7: lane_body<7>(); break; case 8: lane_body<8>(); break; case 9: lane_body<9>(); break; case 10: lane_body<10>(); break;
    }
    wp::emu->done[wp::emu->cur] = true;
    swapcontext(&wp::emu->ctx[wp::emu->cur], &wp::emu->main);
}
template <int NR> long long ws_doubles(int N) { return WarpSolver<NR, NR <= 4>::ws_doubles(N); }   // the larger of the two instantiations
template <int NR> int sm_doubles() { return WarpSolver<NR, NR <= 4>::SM_DOUBLES; }
}  // namespace

extern "C" int emu_solve(const nmpc_desc *d, const nmpc_opts *o, int B, const double *x0, const double *p,
                         const double *lbx, const double *ubx, const double *lbg, const double *ubg,
                         int bounds_batched, double *x, double *f, double *g, double *lam_x, double *lam_g,
                         int *status, int *iters, double *stats, double *trace, int max_trace, int reverse, int nobs, const double *obs)
{
    if (!d || d->Nr < 1 || d->Nr > 10 || d->N < 1) return NMPC_EINVAL;
    const int Nr = d->Nr, N = d->N, S = N + 1, ns = 3 * Nr, nc = 2 * Nr, M = Nr * (Nr - 1) / 2 + Nr * nobs, family = nobs > 0 ? 1 : 0;
    const long long n = (long long)ns * S + (long long)nc * N, mg = family ? ns + (long long)N * (ns + M) : (long long)S * (ns + M);
    const int nb = bounds_batched ? B : 1;
    const int LWd = (5 * Nr + 1 <= 32) ? 32 : 64;
    const long long bstride = (long long)NMPC_BR_COUNT * S * LWd;
    std::vector<double> brows((size_t)nb * bstride);
    int berr = 0;
    for (int b = 0; b < nb; b++)
        for (int k = 0; k < S; k++)
            for (int l = 0; l < LWd; l++) {
                int e = nmpc_prep_bounds_elem(Nr, N, o->bound_relax_factor, lbx + b * n, ubx + b * n, lbg + b * mg,
                                              ubg + b * mg, k, l, LWd, brows.data() + (size_t)b * bstride, nobs, family, 1);
                if (e && !berr) berr = e;
            }
    long long wsd = 0; int smd = 0;
    switch (Nr) {
        case 1: wsd = ws_doubles<1>(N); smd = sm_doubles<1>(); break; case 2: wsd = ws_doubles<2>(N); smd = sm_doubles<2>(); break;
        case 3: wsd = ws_doubles<3>(N); smd = sm_doubles<3>(); break; case 4: wsd = ws_doubles<4>(N); smd = sm_doubles<4>(); break;
        case 5: wsd = ws_doubles<5>(N); smd = sm_doubles<5>(); break; case 6: wsd = ws_doubles<6>(N); smd = sm_doubles<6>(); break;
        case 7: wsd = ws_doubles<7>(N); smd = sm_doubles<7>(); break; case 8: wsd = ws_doubles<8>(N); smd = sm_doubles<8>(); break;
        case 9: wsd = ws_doubles<9>(N); smd = sm_doubles<9>(); break; case 10: wsd = ws_doubles<10>(N); smd = sm_doubles<10>(); break;
    }
    std::vector<double> ws((size_t)wsd, 1e300 /* poison: reads of unwritten scratch must not matter */), sm((size_t)smd, 1e300);
    NmpcSolveParams P;
    memset(&P, 0, sizeof P);
    P.Nr = Nr; P.N = N; P.B = B; P.T = d->T;
    memcpy(P.Q, d->Q, sizeof P.Q); memcpy(P.R, d->R, sizeof P.R);
    P.o = *o; P.x0 = x0; P.p = p; P.brows = brows.data(); P.bstride = bounds_batched ? bstride : 0;
    P.bound_err = &berr; P.x = x; P.f = f; P.g = g; P.lam_x = lam_x; P.lam_g = lam_g; P.status = status; P.iters = iters;
    P.stats = stats; P.trace = trace; P.max_trace = max_trace; P.ws = ws.data(); P.ws_stride = wsd;
    P.np = 6 * Nr;      // p = [x0bar; xs] per instance (the obstacle instantiation strides p by P.np, as nmpc_solve sets it)
    P.nobs = nobs; P.family = family; P.obs = obs;
    const size_t STK = 512 * 1024;
    std::vector<char> stacks(64 * STK);
    wp::Emu emu;
    wp::emu = &emu;
    for (int inst = 0; inst < B; inst++) {
        job.P = &P; job.inst = inst; job.sm = sm.data(); job.ws = ws.data(); job.Nr = Nr;
        for (int l = 0; l < LWd; l++) {
            getcontext(&emu.ctx[l]);
            emu.ctx[l].uc_stack.ss_sp = stacks.data() + (size_t)l * STK;
            emu.ctx[l].uc_stack.ss_size = STK;
            emu.ctx[l].uc_link = &emu.main;
            makecontext(&emu.ctx[l], fibre_main, 0);
            emu.done[l] = false;
        }
        for (;;) {
            bool alive = false;
            for (int i = 0; i < LWd; i++) {
                int l = reverse ? LWd - 1 - i : i;
                if (emu.done[l]) continue;
                alive = true;
                emu.cur = l;
                swapcontext(&emu.main, &emu.ctx[l]);
            }
            if (!alive) break;
        }
    }
    wp::emu = nullptr;
    return berr;
}
