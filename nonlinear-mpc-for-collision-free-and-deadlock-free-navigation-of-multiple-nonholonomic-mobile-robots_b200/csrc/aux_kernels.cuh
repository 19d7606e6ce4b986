// Streaming kernels either side of the solver:
//   K1  eval_kernel   -- stand-alone f, grad f, g, CCS values of dg/dw and of hess(f + lam'g)
//                        (what CasADi's AD sweeps hand IPOPT; NLP of
//                        centralized_six_robots_implementation.py:207-331).  One CTA per point:
//                        w, lam_g, p are loaded coalesced into shared memory, every robot-stage /
//                        pair-stage thread scatters its entries into a shared-memory image of the
//                        output record, and the record is written back with coalesced stores.
//   K4  shift_kernel  -- warm-start shift of the MPC loop (shift() :160-169 and the X0 line :465)
//       plant_kernel  -- Euler plant (casadi_test.py:17-26)
//       prep_bounds_kernel -- flat lbx/ubx/lbg/ubg (:349-352) -> relaxed stage-layout rows
//       advanced_step_kernel -- first-order correction of a solution for the measured state (nmpc_advanced_step)
//       neighbour_kernel -- distributed NMPC: each robot's K nearest teammates' predicted paths as its obstacle block
//                        (nmpc_neighbour_obstacles)
#pragma once
#include "bounds_prep.cuh"
#include "nmpc_internal.h"

// position tables built on the host at nmpc_create (device int arrays)
struct NmpcEvalTables {
    const int *jac_rs;   // [N*Nr*11]  CCS slot of each Jacobian entry of robot-stage (k,i)
    const int *jac_ps;   // [N*M*4]    ... of pair-stage (k,q)
    const int *hes_rs;   // [N*Nr*6]
    const int *hes_ps;   // [N*M*2]
    const int *jac_init; // [ns]       slots of the identity block of the initial-condition rows
};

// All work items of one evaluation point (robot-stage, pair-stage, initial block): fills grad, g and the CCS value arrays of
// the Jacobian and the Hessian of the Lagrangian through the position tables; returns this thread's share of f.  The arrays
// may live in shared memory (eval_kernel: the record is assembled on chip and leaves through bulk stores) or directly in global
// memory (eval_kernel_big: records too large for shared memory, e.g. 2.5 MB at 64 robots); NULL outputs are skipped.
// rstr: stride of the reference in p after x0bar.  0: the setpoint xs (p = [x0bar; xs]); 5 Nr: a tracking handle's
// p = [x0bar; Z[N][5 Nr]], Z[k] = [xr_k; ur_k], whose control reference enters the cost as (U_k - ur_k)' R (U_k - ur_k).
__device__ __forceinline__ double eval_point_items(int Nr, int N, double T, const double *Qw, const double *Rw, const double *sw,
                                                   const double *sl, const double *sp, double *sgrad, double *sg, double *sj,
                                                   double *shs, const NmpcEvalTables &tb, bool lam, bool hess, int rstr)
{
    const int ns = 3 * Nr, nc = 2 * Nr, M = Nr * (Nr - 1) / 2, S = N + 1, blk = ns + M, nX = ns * S;
    double facc = 0.0;
        // robot-stage work items, then pair-stage items, then the initial block
        const int nRS = N * Nr, nPS = N * M;
        for (int it = threadIdx.x; it < nRS + nPS + ns + M + ns; it += blockDim.x) {
            if (it < nRS) {
                const int k = it / Nr, i = it % Nr, r0 = (k + 1) * blk + 3 * i;
                const int ix = k * ns + 3 * i, iu = nX + k * nc + 2 * i;
                const double x = sw[ix], y = sw[ix + 1], th = sw[ix + 2], v = sw[iu], om = sw[iu + 1];
                double s_, c_;
                sincos(th, &s_, &c_);
                const double *rk = sp + ns + k * rstr;
                const double ex = x - rk[3 * i], ey = y - rk[3 * i + 1], et = th - rk[3 * i + 2];
                const double ev = rstr ? v - rk[ns + 2 * i] : v, eo = rstr ? om - rk[ns + 2 * i + 1] : om;
                facc += Qw[0] * ex * ex + Qw[1] * ey * ey + Qw[2] * et * et + Rw[0] * ev * ev + Rw[1] * eo * eo;
                if (sgrad) {
                    sgrad[ix] = 2 * Qw[0] * ex; sgrad[ix + 1] = 2 * Qw[1] * ey; sgrad[ix + 2] = 2 * Qw[2] * et;
                    sgrad[iu] = 2 * Rw[0] * ev; sgrad[iu + 1] = 2 * Rw[1] * eo;
                }
                if (sg) {
                    sg[r0] = sw[ix + ns] - (x + T * v * c_);
                    sg[r0 + 1] = sw[ix + ns + 1] - (y + T * v * s_);
                    sg[r0 + 2] = sw[ix + ns + 2] - (th + T * om);
                }
                const int *js = tb.jac_rs + (size_t)it * 11;
                if (sj) {
                sj[js[0]] = 1.0; sj[js[1]] = -1.0; sj[js[2]] = T * v * s_; sj[js[3]] = -T * c_;
                sj[js[4]] = 1.0; sj[js[5]] = -1.0; sj[js[6]] = -T * v * c_; sj[js[7]] = -T * s_;
                sj[js[8]] = 1.0; sj[js[9]] = -1.0; sj[js[10]] = -T;
                }
                if (lam && hess && shs) {
                    const double lx = sl[r0], ly = sl[r0 + 1];
                    double sm2 = 0.0;
                    for (int j = 0; j < Nr; j++) {
                        if (j == i) continue;
                        const int a = i < j ? i : j, c2 = i < j ? j : i;
                        sm2 += 2.0 * sl[(k + 1) * blk + ns + a * (2 * Nr - a - 1) / 2 + (c2 - a - 1)];
                    }
                    const int *hs = tb.hes_rs + (size_t)it * 6;
                    shs[hs[0]] = 2 * Qw[0] + sm2; shs[hs[1]] = 2 * Qw[1] + sm2;
                    shs[hs[2]] = 2 * Qw[2] + T * v * (lx * c_ + ly * s_);
                    shs[hs[3]] = T * (lx * s_ - ly * c_);
                    shs[hs[4]] = 2 * Rw[0]; shs[hs[5]] = 2 * Rw[1];
                }
            } else if (it < nRS + nPS) {
                const int e = it - nRS, k = e / M, q = e % M;
                int a = 0, rem = q;
                while (rem >= Nr - 1 - a) { rem -= Nr - 1 - a; a++; }
                const int c2 = a + 1 + rem;
                const double dx = sw[k * ns + 3 * a] - sw[k * ns + 3 * c2], dy = sw[k * ns + 3 * a + 1] - sw[k * ns + 3 * c2 + 1];
                if (sg) sg[(k + 1) * blk + ns + q] = dx * dx + dy * dy;
                const int *js = tb.jac_ps + (size_t)e * 4;
                if (sj) { sj[js[0]] = 2 * dx; sj[js[1]] = -2 * dx; sj[js[2]] = 2 * dy; sj[js[3]] = -2 * dy; }
                if (lam && hess && shs) {
                    const double mu = sl[(k + 1) * blk + ns + q];
                    const int *hs = tb.hes_ps + (size_t)e * 2;
                    shs[hs[0]] = -2 * mu; shs[hs[1]] = -2 * mu;
                }
            } else if (it < nRS + nPS + ns) {
                const int r = it - nRS - nPS;
                if (sg) sg[r] = sw[r] - sp[r];
                if (sj) sj[tb.jac_init[r]] = 1.0;
            } else if (it < nRS + nPS + ns + M) {
                if (sg) sg[ns + (it - nRS - nPS - ns)] = NMPC_DUMMY_ROW_VALUE;
            } else {
                if (sgrad) sgrad[N * ns + (it - nRS - nPS - ns - M)] = 0.0;  // X_N is not in the cost
            }
        }
    return facc;
}

// TMA bulk store shared -> global (cp.async.bulk, one elected thread issues it; completion tracked per bulk group)
__device__ __forceinline__ void bulk_store_s2g(void *gdst, const void *ssrc, unsigned bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"((unsigned)__cvta_generic_to_shared(ssrc)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// TRK: a tracking handle's p (np = 3 Nr + 5 Nr N = n, so the prefetch of p takes PF registers like w); else p = [x0bar; xs]
template <int PF, bool TRK>
__global__ void __launch_bounds__(256) eval_kernel(int Nr, int N, double T, double Q0, double Q1, double Q2, double R0,
                                                   double R1, int B, const double *__restrict__ w, const double *__restrict__ p,
                                                   const double *__restrict__ lam, double *__restrict__ f, double *__restrict__ grad,
                                                   double *__restrict__ g, double *__restrict__ jac, double *__restrict__ hess,
                                                   NmpcEvalTables tb)
{
    extern __shared__ double sh[];
    const int ns = 3 * Nr, nc = 2 * Nr, M = Nr * (Nr - 1) / 2, S = N + 1, blk = ns + M;
    const int n = ns * S + nc * N, mg = S * blk, nX = ns * S;
    const int nj = 3 * Nr + N * (11 * Nr + 4 * M), nh = N * (6 * Nr + 2 * M);
    const int np = TRK ? ns + N * (ns + nc) : 2 * ns, rstr = TRK ? ns + nc : 0;
    auto ev = [](int v) { return (v + 1) & ~1; };   // every segment starts 16-byte aligned (128-bit write-back)
    double *sw = sh, *sl = sw + ev(n), *sp = sl + ev(mg), *sgrad = sp + ev(np), *sg0 = sgrad + ev(n), *sj = sg0 + ev(mg + 1),
           *shs = sj + ev(nj), *sred = shs + ev(nh);
    const double Qw[3] = {Q0, Q1, Q2}, Rw[2] = {R0, R1};
    // The inputs of the next point are fetched into PF registers per array per thread right after the evaluation of
    // the current point, so their HBM latency overlaps the write-back (PF = ceil(max(n, mg) / 256), 0 = no prefetch).
    double rw[PF > 0 ? PF : 1], rl[PF > 0 ? PF : 1], rq[(TRK && PF > 0) ? PF : 1], rp = 0.0;
    auto fetch = [&](int b) {
        if (PF == 0 || b >= B) return;
#pragma unroll
        for (int j = 0; j < PF; j++) {
            const int i = threadIdx.x + j * 256;
            rw[j] = i < n ? w[(size_t)b * n + i] : 0.0;
            rl[j] = (lam && i < mg) ? lam[(size_t)b * mg + i] : 0.0;
            if (TRK) rq[j] = i < np ? p[(size_t)b * np + i] : 0.0;
        }
        if (!TRK) rp = (int)threadIdx.x < 2 * ns ? p[(size_t)b * 2 * ns + threadIdx.x] : 0.0;
    };
    fetch(blockIdx.x);
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        // g has an odd length at Nr = 6 (mg = 693): its shared copy starts 8 bytes in whenever the global segment does,
        // so that all but its first / last element can leave through an aligned bulk store as well
        double *sg = sg0 + ((g && (((size_t)(g + (size_t)b * mg)) & 15)) ? 1 : 0);
        if (PF > 0) {
#pragma unroll
            for (int j = 0; j < PF; j++) {
                const int i = threadIdx.x + j * 256;
                if (i < n) sw[i] = rw[j];
                if (lam && i < mg) sl[i] = rl[j];
                if (TRK && i < np) sp[i] = rq[j];
            }
            if (!TRK && (int)threadIdx.x < 2 * ns) sp[threadIdx.x] = rp;
            if (threadIdx.x == 0) bulk_wait_read_all();   // the previous point's bulk stores have finished reading the record
        } else {
            if (threadIdx.x == 0) bulk_wait_read_all();
            const double *wb = w + (size_t)b * n;
            for (int i = threadIdx.x; i < n; i += blockDim.x) sw[i] = wb[i];
            for (int i = threadIdx.x; i < np; i += blockDim.x) sp[i] = p[(size_t)b * np + i];
            if (lam) for (int i = threadIdx.x; i < mg; i += blockDim.x) sl[i] = lam[(size_t)b * mg + i];
        }
        __syncthreads();
        double facc = eval_point_items(Nr, N, T, Qw, Rw, sw, sl, sp, sgrad, sg, sj, shs, tb, lam != nullptr, hess != nullptr,
                                       rstr);
        // block reduction of f
        for (int m = 16; m > 0; m >>= 1) facc += __shfl_xor_sync(0xffffffffu, facc, m);
        if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = facc;
        fence_proxy_async_smem();   // the record written above becomes visible to the bulk-copy engine
        __syncthreads();
        if (threadIdx.x == 0 && f) {
            double t = 0.0;
            for (int i = 0; i < (int)(blockDim.x >> 5); i++) t += sred[i];
            f[b] = t;
        }
        fetch(b + gridDim.x);   // next point's inputs: in flight during the write-back below
        // write-back of the record: segments that are 16-byte aligned with an even length leave through ONE TMA bulk
        // store each (cp.async.bulk shared -> global, issued by thread 0, asynchronous: the CTA goes on to the next point
        // and only waits, above, until the engine has read the record); the others (g: mg is odd at Nr = 6) through
        // coalesced stores, 128-bit where possible
        auto copy_out = [&](double *dst, const double *src, int cnt) {
            if (!dst) return;
            if ((((size_t)dst ^ (size_t)src) & 15) == 0 && (((size_t)dst) & 7) == 0) {
                // same 16-byte phase on both sides: scalar head / tail, aligned bulk body
                const int head = (((size_t)dst) & 15) ? 1 : 0, body = (cnt - head) & ~1, tail = cnt - head - body;
                if (threadIdx.x == 0) {
                    if (head) dst[0] = src[0];
                    if (body) bulk_store_s2g(dst + head, src + head, (unsigned)body * 8u);
                    if (tail) dst[cnt - 1] = src[cnt - 1];
                }
            } else if ((((size_t)dst | (size_t)src) & 15) == 0) {
                const int c2 = cnt >> 1;
                double2 *d2 = reinterpret_cast<double2 *>(dst);
                const double2 *s2 = reinterpret_cast<const double2 *>(src);
                for (int i = threadIdx.x; i < c2; i += blockDim.x) d2[i] = s2[i];
                if ((cnt & 1) && threadIdx.x == 0) dst[cnt - 1] = src[cnt - 1];
            } else {
                for (int i = threadIdx.x; i < cnt; i += blockDim.x) dst[i] = src[i];
            }
        };
        copy_out(grad ? grad + (size_t)b * n : nullptr, sgrad, n);
        copy_out(g ? g + (size_t)b * mg : nullptr, sg, mg);
        copy_out(jac ? jac + (size_t)b * nj : nullptr, sj, nj);
        copy_out((hess && lam) ? hess + (size_t)b * nh : nullptr, shs, nh);
        if (threadIdx.x == 0) bulk_commit();
        __syncthreads();
    }
    if (threadIdx.x == 0) bulk_wait_read_all();   // shared memory must outlive the last bulk stores
}

// Records that do not fit shared memory (more than ~11 robots at N = 20): same work items, written straight to global memory.
// np, rstr: width of p and stride of its reference (see eval_point_items)
__global__ void __launch_bounds__(256) eval_kernel_big(int Nr, int N, double T, double Q0, double Q1, double Q2, double R0, double R1, int B,
                                                       const double *__restrict__ w, const double *__restrict__ p,
                                                       const double *__restrict__ lam, double *__restrict__ f, double *__restrict__ grad,
                                                       double *__restrict__ g, double *__restrict__ jac, double *__restrict__ hess,
                                                       NmpcEvalTables tb, int np, int rstr)
{
    __shared__ double sred[8];
    const int ns = 3 * Nr, nc = 2 * Nr, M = Nr * (Nr - 1) / 2, S = N + 1;
    const size_t n = (size_t)ns * S + (size_t)nc * N, mg = (size_t)S * (ns + M);
    const size_t nj = 3 * (size_t)Nr + (size_t)N * (11 * Nr + 4 * M), nh = (size_t)N * (6 * Nr + 2 * M);
    const double Qw[3] = {Q0, Q1, Q2}, Rw[2] = {R0, R1};
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        double facc = eval_point_items(Nr, N, T, Qw, Rw, w + b * n, lam ? lam + b * mg : nullptr, p + (size_t)b * np,
                                       grad ? grad + b * n : nullptr, g ? g + b * mg : nullptr, jac ? jac + b * nj : nullptr,
                                       hess ? hess + b * nh : nullptr, tb, lam != nullptr, hess != nullptr, rstr);
        for (int m = 16; m > 0; m >>= 1) facc += __shfl_xor_sync(0xffffffffu, facc, m);
        if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = facc;
        __syncthreads();
        if (threadIdx.x == 0 && f) {
            double t = 0.0;
            for (int i = 0; i < (int)(blockDim.x >> 5); i++) t += sred[i];
            f[b] = t;
        }
        __syncthreads();
    }
}

// u0 = [u[1:]; u[-1]]  and  X0 = [X[1:]; X[N-1]]   (row N-1, not N: the reference's quirk)
__global__ void __launch_bounds__(256) shift_kernel(int Nr, int N, long long total, const double *__restrict__ xp, double *__restrict__ xn)
{
    // one instance per CTA iteration; the source index is piecewise linear in the destination index:
    //   states   j <  ns*N        -> j + ns          (X_{k+1})
    //            j in last block  -> j - ns          (X_{N-1}: the reference appends row N-1, not N)
    //   controls j <  nc*(N-1)    -> j + nc          (U_{k+1})
    //            last block       -> j               (U_{N-1} repeated)
    const int ns = 3 * Nr, nc = 2 * Nr, nX = ns * (N + 1), n = nX + nc * N;
    const long long B = total / n;
    // every segment boundary (ns, nc, nX, n) is even when Nr is even: the copy then runs on 128-bit loads and stores
    const bool vec = ((ns | nc | n) & 1) == 0 && ((((size_t)xp) | ((size_t)xn)) & 15) == 0;
    if (vec) {   // flat grid-stride loop over all 128-bit elements of the batch: full warps whatever n is
        const int n2 = n / 2;
        const long long total2 = B * n2;
        const double2 *s2 = reinterpret_cast<const double2 *>(xp);
        double2 *d2 = reinterpret_cast<double2 *>(xn);
        for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total2; e += (long long)gridDim.x * blockDim.x) {
            const long long b = e / n2;
            const int j = 2 * (int)(e - b * n2);
            int s;
            if (j < nX) s = j < ns * N ? j + ns : j - ns;
            else s = (j - nX) < nc * (N - 1) ? j + nc : j;
            d2[e] = s2[b * n2 + (s >> 1)];
        }
        return;
    }
    for (long long b = blockIdx.x; b < B; b += gridDim.x) {
        const double *src = xp + b * n;
        double *dst = xn + b * n;
        for (int j = threadIdx.x; j < n; j += blockDim.x) {
            int s;
            if (j < nX) s = j < ns * N ? j + ns : j - ns;
            else s = (j - nX) < nc * (N - 1) ? j + nc : j;
            dst[j] = src[s];
        }
    }
}

__global__ void plant_kernel(int Nr, int N, double T, int B, const double *__restrict__ st, const double *__restrict__ xopt,
                             double *__restrict__ out)
{
    const int ns = 3 * Nr, nc = 2 * Nr, nX = ns * (N + 1), n = nX + nc * N;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < B * Nr; e += gridDim.x * blockDim.x) {
        const int b = e / Nr, i = e % Nr;
        const double *s = st + (size_t)b * ns + 3 * i;
        const double v = xopt[(size_t)b * n + nX + 2 * i], om = xopt[(size_t)b * n + nX + 2 * i + 1];
        const double x = s[0], y = s[1], th = s[2];
        double s_, c_;
        sincos(th, &s_, &c_);
        double *o = out + (size_t)b * ns + 3 * i;
        o[0] = x + T * v * c_; o[1] = y + T * v * s_; o[2] = th + T * om;
    }
}

__global__ void prep_bounds_kernel(int Nr, int N, double relax, int nb, int lw, const double *__restrict__ lbx, const double *__restrict__ ubx,
                                   const double *__restrict__ lbg, const double *__restrict__ ubg, double *__restrict__ rows, int *err,
                                   int nobs = 0, int family = 0, int stage_major = 0)
{
    const int S = N + 1, ns = 3 * Nr, nc = 2 * Nr, M = Nr * (Nr - 1) / 2 + Nr * nobs;
    const long long n = (long long)ns * S + (long long)nc * N, mg = family ? ns + (long long)N * (ns + M) : (long long)S * (ns + M);
    const long long total = (long long)nb * S * lw, bstride = (long long)NMPC_BR_COUNT * S * lw;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long b = e / (S * lw);
        const int k = (int)((e / lw) % S), lane = (int)(e % lw);
        int rc = nmpc_prep_bounds_elem(Nr, N, relax, lbx + b * n, ubx + b * n, lbg + b * mg, ubg + b * mg, k, lane, lw, rows + b * bstride, nobs, family, stage_major);
        if (rc) atomicCAS(err, 0, rc);
    }
}

// Advanced-step feedback (nmpc_advanced_step): x_corr = x + jac' (x0bar_meas - p[0:ns]) per instance, one thread per (instance,
// variable), jac [B][ns][n] read coalesced along n; the sum runs over j = 0..ns-1 in order.  A variable with a finite bound is
// clamped to [min(lb, x), max(ub, x)], so a component the solve left just outside its bound (bound_relax_factor) is never pulled
// further; the X_0 rows are x0bar_meas exactly.  An instance with sens_status != 0 keeps x (X_0 = x0bar_meas all the same).
__global__ void __launch_bounds__(256) advanced_step_kernel(int ns, int n, int np, long long total, const double *__restrict__ x,
                                                            const double *__restrict__ jac, const int *__restrict__ sens_status,
                                                            const double *__restrict__ p, const double *__restrict__ x0m,
                                                            const double *__restrict__ lbx, const double *__restrict__ ubx,
                                                            long long bstride, double *__restrict__ xc)
{
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long b = e / n;
        const int i = (int)(e - b * n);
        const double *meas = x0m + b * ns;
        if (i < ns) { xc[e] = meas[i]; continue; }
        const double xi = x[e];
        if (sens_status[b] != 0) { xc[e] = xi; continue; }
        const double *jb = jac + b * ns * n + i, *pb = p + b * np;
        double s = 0.0;
        for (int j = 0; j < ns; j++) s = fma(jb[(long long)j * n], meas[j] - pb[j], s);
        double v = xi + s;
        const double lb = lbx[b * bstride + i], ub = ubx[b * bstride + i];
        if (lb > -NMPC_INF) v = fmax(v, fmin(lb, xi));
        if (ub < NMPC_INF) v = fmin(v, fmax(ub, xi));
        xc[e] = v;
    }
}

// Neighbour exchange of distributed NMPC (nmpc_neighbour_obstacles).  Robot j's prediction at stage k < N is its pose state[j] at
// k = 0 and X_{min(k+1, N)} of its plan (plan [S R][n], X_k at 3k) for k >= 1: the plan shifted by one period with the last stage
// repeated; plan == NULL holds the pose at every stage.  For robot a the key of a teammate j != a of its scenario is (d2, j),
// d2 = min over k < N of the squared xy distance of the two predictions; the K smallest keys in lexicographic order (ties to the
// lower index) give O[k][o] = (x, y, clearance) of the o-th one at stage k, and a slot left without a teammate (R - 1 < K) gets an
// inactive obstacle: the own pose + (1e6, 0) with clearance 0.  x0bar = state; nothing else of p is written.  min_dist[a] is the
// distance from a's pose to the nearest other robot of its scenario (+inf for R = 1).
// One warp per robot, NB_WARPS robots of one scenario per CTA, (scenario, robot group) pairs strided over the grid.  Tiles of 32
// candidates x N stages are staged in shared memory once per CTA for all its warps, stage-major ([N][32] double2, so lane c reads
// its candidate's stage k without bank conflicts); each lane computes one candidate's key, and the warp keeps its 32 smallest keys
// sorted across its lanes: a bitonic network on shuffles sorts the tile's 32 keys, min(kept[l], new[31 - l]) leaves the 32
// smallest of the 64 as a bitonic sequence, and a 5-step bitonic merge sorts them again.  The arithmetic is __dsub_rn / __dmul_rn /
// __dadd_rn (no FMA contraction), fmin and a correctly rounded sqrt, so a NumPy restatement matches bit for bit, and the result
// depends neither on the tiling nor on the lane order (the keys are distinct but for the padding key, which is one value).
#define NB_WARPS 8
#define NB_NONE 0x7fffffff   // index of the padding key
struct NbKey { double d; int j; };
__device__ __forceinline__ bool nb_less(const NbKey &a, const NbKey &b) { return a.d < b.d || (a.d == b.d && a.j < b.j); }
// compare-exchange with lane ^ m: the smaller of the two keys if keep_min, else the larger
__device__ __forceinline__ NbKey nb_cx(const NbKey &k, int m, bool keep_min)
{
    const NbKey o = {__shfl_xor_sync(0xffffffffu, k.d, m), __shfl_xor_sync(0xffffffffu, k.j, m)};
    return nb_less(o, k) == keep_min ? o : k;
}

__global__ void __launch_bounds__(NB_WARPS * 32) neighbour_kernel(int N, int K, int S, int R, int n, int np,
                                                                  const double *__restrict__ state, const double *__restrict__ plan,
                                                                  double clearance, double *__restrict__ p, double *__restrict__ min_dist)
{
    extern __shared__ double2 nb_sh[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double2 *tile = nb_sh, *own = nb_sh + (size_t)N * 32 + (size_t)warp * N;   // [N][32] candidates, [N] this warp's robot
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    const int groups = (R + NB_WARPS - 1) / NB_WARPS;
    auto pred = [&](long long j, int k) {
        const double *s = (k == 0 || !plan) ? state + 3 * j : plan + j * n + 3 * min(k + 1, N);
        return make_double2(s[0], s[1]);
    };
    for (long long g = blockIdx.x; g < (long long)S * groups; g += gridDim.x) {
        const long long base = (g / groups) * R;
        const int a = (int)(g % groups) * NB_WARPS + warp;
        const bool live = a < R;   // uniform over the warp
        __syncwarp();
        if (live)
            for (int k = lane; k < N; k += 32) own[k] = pred(base + a, k);
        NbKey kept = {inf, NB_NONE};
        double d0 = inf;   // smallest squared distance between current poses seen by this lane
        for (int j0 = 0; j0 < R; j0 += 32) {
            __syncthreads();   // every warp is done with the previous tile
            for (int e = threadIdx.x; e < 32 * N; e += blockDim.x)
                if (j0 + (e & 31) < R) tile[e] = pred(base + j0 + (e & 31), e >> 5);
            __syncthreads();
            const int j = j0 + lane;
            NbKey nk = {inf, NB_NONE};
            if (live && j < R && j != a) {
                double dm = inf;
                for (int k = 0; k < N; k++) {
                    const double2 q = tile[k * 32 + lane], o = own[k];
                    const double dx = __dsub_rn(o.x, q.x), dy = __dsub_rn(o.y, q.y);
                    const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
                    if (k == 0) d0 = fmin(d0, d2);
                    dm = fmin(dm, d2);
                }
                nk = {dm, j};
            }
#pragma unroll
            for (int size = 2; size <= 32; size <<= 1)
#pragma unroll
                for (int m = size >> 1; m > 0; m >>= 1) nk = nb_cx(nk, m, ((lane & m) == 0) == ((lane & size) == 0));
            const NbKey r = {__shfl_sync(0xffffffffu, nk.d, 31 - lane), __shfl_sync(0xffffffffu, nk.j, 31 - lane)};
            if (nb_less(r, kept)) kept = r;
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) kept = nb_cx(kept, m, (lane & m) == 0);
        }
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) d0 = fmin(d0, __shfl_xor_sync(0xffffffffu, d0, m));
        if (!live) continue;
        const long long ia = base + a;
        double *pa = p + ia * np, *O = pa + (np - 3 * N * K);
        if (lane < 3) pa[lane] = state[3 * ia + lane];
        if (lane == 0 && min_dist) min_dist[ia] = sqrt(d0);
        const double2 me = own[0];
        for (int e0 = 0; e0 < N * K; e0 += 32) {   // entry e = (k, o) = (e / K, e % K) of the block, three doubles each
            const int e = e0 + lane, jo = __shfl_sync(0xffffffffu, kept.j, e % K);
            if (e >= N * K) continue;
            double2 q = make_double2(__dadd_rn(me.x, 1e6), me.y);
            double c = 0.0;
            if (jo != NB_NONE) { q = pred(base + jo, e / K); c = clearance; }
            O[3 * e] = q.x; O[3 * e + 1] = q.y; O[3 * e + 2] = c;
        }
    }
}
