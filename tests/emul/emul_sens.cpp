// CPU fibre emulation of the product's sensitivity pass (WarpSolver::sensitivity, nmpc_solution_vjp / _jvp) -- TEST
// INFRASTRUCTURE ONLY.  Compiles csrc/solver_body.cuh (unchanged) against tests/emul/warp_prims.cuh, like emul_solver.cpp;
// SENS_TRK selects the tracking instantiation.  Scratch and shared memory are poisoned (1e300) before every instance.
#include "warp_prims.cuh"
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "solver_body.cuh"
#include "bounds_prep.cuh"

#ifndef SENS_TRK
#define SENS_TRK 0
#endif

namespace wp { thread_local Emu *emu = nullptr; }

namespace {
struct Job { const NmpcSolveParams *P; const NmpcSensParams *S; int inst; double *sm, *ws; int Nr; };
thread_local Job job;

template <int NR> void lane_body()
{
    WarpSolver<NR, false, SENS_TRK> s(*job.P, job.sm, job.ws);
    s.init_team();
    s.setup(job.inst);
    s.sensitivity(*job.S);
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
template <int NR> long long ws_doubles(int N) { return WarpSolver<NR, false, SENS_TRK>::ws_doubles(N); }
template <int NR> int sm_doubles() { return WarpSolver<NR, false, SENS_TRK>::SM_DOUBLES; }
}  // namespace

// reverse = 1: seed x_bar [B,n] -> out p_bar [B,np];  0: seed p_dot [B,np] -> out x_dot [B,n].  lane_rev: lanes in reverse order.
extern "C" int emu_sens(const nmpc_desc *d, const nmpc_opts *o, int B, const double *x, const double *lam_x, const double *lam_g,
                        const double *p, const double *lbx, const double *ubx, const double *lbg, const double *ubg,
                        int bounds_batched, const double *seed, double *out, int *status, int reverse, int lane_rev)
{
    if (!d || d->Nr < 1 || d->Nr > 10 || d->N < 1) return NMPC_EINVAL;
    const int Nr = d->Nr, N = d->N, S = N + 1, ns = 3 * Nr, nc = 2 * Nr, M = Nr * (Nr - 1) / 2;
    const long long n = (long long)ns * S + (long long)nc * N, mg = (long long)S * (ns + M);
    const int nb = bounds_batched ? B : 1;
    const int LWd = (5 * Nr + 1 <= 32) ? 32 : 64;
    const long long bstride = (long long)NMPC_BR_COUNT * S * LWd;
    std::vector<double> brows((size_t)nb * bstride);
    int berr = 0;
    for (int b = 0; b < nb; b++)
        for (int k = 0; k < S; k++)
            for (int l = 0; l < LWd; l++) {
                int e = nmpc_prep_bounds_elem(Nr, N, o->bound_relax_factor, lbx + b * n, ubx + b * n, lbg + b * mg,
                                              ubg + b * mg, k, l, LWd, brows.data() + (size_t)b * bstride, 0, 0, 1);
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
    std::vector<double> ws((size_t)wsd), sm((size_t)smd);
    NmpcSolveParams P;
    memset(&P, 0, sizeof P);
    P.Nr = Nr; P.N = N; P.B = B; P.T = d->T;
    memcpy(P.Q, d->Q, sizeof P.Q); memcpy(P.R, d->R, sizeof P.R);
    P.o = *o; P.p = p; P.brows = brows.data(); P.bstride = bounds_batched ? bstride : 0;
    P.bound_err = &berr; P.ws = ws.data(); P.ws_stride = wsd;
    P.np = SENS_TRK ? ns + N * (ns + nc) : 2 * ns;
    NmpcSensParams SP;
    SP.x = x; SP.lam_x = lam_x; SP.lam_g = lam_g; SP.seed = seed; SP.out = out; SP.status = status; SP.reverse = reverse;
    const size_t STK = 512 * 1024;
    std::vector<char> stacks(64 * STK);
    wp::Emu emu;
    wp::emu = &emu;
    for (int inst = 0; inst < B; inst++) {
        for (auto &v : ws) v = 1e300;   // poison: reads of scratch the pass did not write must not matter
        for (auto &v : sm) v = 1e300;
        job.P = &P; job.S = &SP; job.inst = inst; job.sm = sm.data(); job.ws = ws.data(); job.Nr = Nr;
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
                int l = lane_rev ? LWd - 1 - i : i;
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
