"""References of the streaming kernels either side of the solver (K1 nmpc_eval, nmpc_shift, nmpc_plant, nmpc_advanced_step)
for tests/test_streaming_kernels.py -- TEST INFRASTRUCTURE ONLY.

EvalRef restates the K1 record (f, grad f, g, and the CCS values of dg/dw and of the lower triangle of hess(f + lam'g)) over a
whole batch at once, for both layouts of p: [x0bar; xs] and the tracking [x0bar; Z[N][5 Nr]].  The (row, col) of every CCS slot
is taken from the pattern the handle reports, and the closed-form partial of that entry is evaluated for all points; dense
per-point matrices would not fit at the batch sizes the kernels run at.  Next to every value it returns S, the sum of the
absolute values of the terms of its expression, so that a device value can be held to |dev - ref| <= k eps S.  The same code
runs on float64 arrays and on object arrays of mpmath numbers (sin / cos passed in), which is how its own rounding error is
measured.

eval_launch mirrors the launch selection of nmpc_eval (csrc/nmpc_b200.cu): which of the 20 kernels runs and on how many CTAs.
Nothing on the device reports the instantiation that ran, so this mirror is the coverage record of the tests.
"""
import math

import numpy as np

EPS = np.finfo(np.float64).eps
DUMMY_ROW = 3.5              # NMPC_DUMMY_ROW_VALUE (csrc/nmpc_internal.h): the stage-0 pair rows
SMEM_CAP = 220 * 1024        # the eval record budget of shared memory per CTA
BIG_CTAS_PER_SM = 8


def dims(Nr, N, tracking):
    ns, nc, M = 3 * Nr, 2 * Nr, Nr * (Nr - 1) // 2
    return dict(ns=ns, nc=nc, M=M, blk=ns + M, nX=ns * (N + 1), n=ns * (N + 1) + nc * N, mg=(N + 1) * (ns + M),
                np=ns + N * (ns + nc) if tracking else 2 * ns, nnzj=3 * Nr + N * (11 * Nr + 4 * M), nnzh=N * (6 * Nr + 2 * M))


def eval_launch(Nr, N, tracking, sm_count, B=None):
    """(variant, grid, eval_smem) of nmpc_eval for a handle of this shape: variant is PF = 0..8 of eval_kernel<PF, TRK> or
    'big' for eval_kernel_big.  Mirrors csrc/nmpc_b200.cu:
      create_impl   :446  eval_smem = (2 n + 2 mg + np + nnz_jac + nnz_hess + 32 + 8) doubles
                    :358, :447  eval_ok = family 0 and eval_smem <= 220 KiB
      nmpc_eval     :877  eval_ok false: eval_kernel_big on min(B, 8 sm_count) CTAs
                    :884  per_sm = max(1, 220 KiB / eval_smem);  :885  grid = min(B, sm_count per_sm)
                    :886, :896  PF = ceil(max(n, mg) / 256), PF > 8 -> 0 (no register prefetch)
    B = None: the grid of a batch at least that large."""
    d = dims(Nr, N, tracking)
    smem = (2 * d["n"] + 2 * d["mg"] + d["np"] + d["nnzj"] + d["nnzh"] + 32 + 8) * 8
    if smem > SMEM_CAP:
        variant, grid = "big", sm_count * BIG_CTAS_PER_SM
    else:
        pf = (max(d["n"], d["mg"]) + 255) // 256
        variant, grid = (pf if pf <= 8 else 0), sm_count * max(1, SMEM_CAP // smem)
    return variant, (grid if B is None else min(B, grid)), smem


def _decode_var(j, ns, nc, nX):
    """Column j of w -> (is_state, stage, robot, component)."""
    if j < nX:
        return True, j // ns, (j % ns) // 3, j % 3
    u = j - nX
    return False, u // nc, (u % nc) // 2, u % 2


class EvalRef:
    """The K1 record of a (Nr, N, T, Q, R) handle, setpoint or tracking, with slots ordered as jac_pattern / hess_pattern."""

    def __init__(self, Nr, N, T, Q, R, tracking, jac_pattern, hess_pattern):
        self.Nr, self.N, self.T, self.tracking = int(Nr), int(N), float(T), bool(tracking)
        self.Q, self.R = tuple(float(q) for q in Q), tuple(float(r) for r in R)
        self.d = d = dims(Nr, N, tracking)
        ns, nc, M, blk, nX = d["ns"], d["nc"], d["M"], d["blk"], d["nX"]
        self.pairs = [(a, b) for a in range(Nr) for b in range(a + 1, Nr)]
        pidx = {ab: q for q, ab in enumerate(self.pairs)}
        # Jacobian: slot -> kind; robot-stage kinds gather from [B, N Nr] tables at k Nr + i, pair kinds from [B, N M] at k M + q
        cp, ri = (np.asarray(a) for a in jac_pattern)
        assert len(cp) == d["n"] + 1 and len(ri) == d["nnzj"]
        jk = {}
        for j in range(d["n"]):
            st, kc, ic, cc = _decode_var(j, ns, nc, nX)
            for s in range(cp[j], cp[j + 1]):
                r = int(ri[s])
                kb, l = divmod(r, blk)
                if kb == 0:
                    assert l < ns and j == r, (r, j)
                    key, at = ("c", 1.0), 0
                elif l < ns:
                    k, i, c = kb - 1, l // 3, l % 3
                    at = k * Nr + i
                    if st and kc == k + 1 and (ic, cc) == (i, c):
                        key = ("c", 1.0)
                    elif st and kc == k and ic == i and cc == c:
                        key = ("c", -1.0)
                    elif st and kc == k and ic == i and cc == 2:
                        key = {0: "Tvs", 1: "mTvc"}[c]
                    elif not st and kc == k and ic == i:
                        key = {(0, 0): "mTc", (1, 0): "mTs", (2, 1): ("c", -self.T)}[(c, cc)]
                    else:
                        raise AssertionError("Jacobian slot (%d, %d) has no partial" % (r, j))
                else:
                    k, q = kb - 1, l - ns
                    a, b = self.pairs[q]
                    assert st and kc == k and cc in (0, 1) and ic in (a, b), (r, j)
                    key, at = ("p%s%d" % ("m" if ic == b else "", cc), k * M + q)
                jk.setdefault(key, ([], []))
                jk[key][0].append(s)
                jk[key][1].append(at)
        self.jac_kinds = {k: (np.array(v[0]), np.array(v[1])) for k, v in jk.items()}
        # Hessian of the Lagrangian, lower triangle
        cp, ri = (np.asarray(a) for a in hess_pattern)
        assert len(cp) == d["n"] + 1 and len(ri) == d["nnzh"]
        hk = {}
        for j in range(d["n"]):
            sc, kc, ic, cc = _decode_var(j, ns, nc, nX)
            for s in range(cp[j], cp[j + 1]):
                r = int(ri[s])
                sr, kr, ir, cr = _decode_var(r, ns, nc, nX)
                assert r >= j and kr == kc and kc < N, (r, j)
                if r == j:
                    key = ("xx", "yy", "tt")[cc] if sc else ("c", 2.0 * self.R[cc])
                    at = kc * Nr + ic
                elif sc and not sr and ir == ic and (cc, cr) == (2, 0):
                    key, at = "vt", kc * Nr + ic
                elif sc and sr and cr == cc and cc in (0, 1) and ir != ic:
                    key, at = "mu", kc * M + pidx[(min(ir, ic), max(ir, ic))]
                else:
                    raise AssertionError("Hessian slot (%d, %d) has no partial" % (r, j))
                hk.setdefault(key, ([], []))
                hk[key][0].append(s)
                hk[key][1].append(at)
        self.hess_kinds = {k: (np.array(v[0]), np.array(v[1])) for k, v in hk.items()}

    def eval(self, W, P, LAM, sin=np.sin, cos=np.cos):
        """Record of the points W [B, n], P [B, np], LAM [B, mg] (or None: no Hessian).  Returns {name: (value, S)}; f also
        carries its number of terms: ('f': (f, S, n_terms)).  float64 arrays, or object arrays of mpmath numbers together with
        elementwise sin / cos for those."""
        d, Nr, N, T = self.d, self.Nr, self.N, self.T
        ns, nc, M, blk, nX = d["ns"], d["nc"], d["M"], d["blk"], d["nX"]
        B = W.shape[0]
        exact = W.dtype == object
        X = W[:, :nX].reshape(B, N + 1, Nr, 3)
        U = W[:, nX:].reshape(B, N, Nr, 2)
        if self.tracking:
            Z = P[:, ns:ns + N * (ns + nc)].reshape(B, N, ns + nc)
            xr, ur = Z[:, :, :ns].reshape(B, N, Nr, 3), Z[:, :, ns:].reshape(B, N, Nr, 2)
            e, eu = X[:, :N] - xr, U - ur
        else:
            e, eu = X[:, :N] - P[:, None, ns:2 * ns].reshape(B, 1, Nr, 3), U
        th, v, om = X[:, :N, :, 2], U[..., 0], U[..., 1]
        sn, cs = sin(th), cos(th)
        Qv, Rv = np.array(self.Q, dtype=W.dtype), np.array(self.R, dtype=W.dtype)
        out = {}
        # f: the kernel's facc += Q0 ex ex + ... , as separate terms summed exactly
        terms = np.concatenate([(Qv * e * e).reshape(B, -1), (Rv * eu * eu).reshape(B, -1)], axis=1)
        fsum = (lambda r: sum(r)) if exact else math.fsum
        out["f"] = (np.array([fsum(r) for r in terms], dtype=W.dtype), np.abs(terms).sum(axis=1), terms.shape[1])
        # grad f: 2 Q e on X_0..X_{N-1}, 0 on X_N, 2 R (U - ur)
        gX = np.zeros((B, N + 1, Nr, 3), dtype=W.dtype)
        gX[:, :N] = (2 * Qv) * e
        grad = np.concatenate([gX.reshape(B, -1), ((2 * Rv) * eu).reshape(B, -1)], axis=1)
        out["grad"] = (grad, np.abs(grad))
        # g: [X_0 - x0bar; dummy pair rows], then per stage [X_{k+1} - (X_k + T f(X_k, U_k)); squared pair distances]
        g = np.zeros((B, N + 1, blk), dtype=W.dtype)
        gS = np.zeros((B, N + 1, blk), dtype=W.dtype)
        g[:, 0, :ns] = W[:, :ns] - P[:, :ns]
        gS[:, 0, :ns] = np.abs(W[:, :ns]) + np.abs(P[:, :ns])
        g[:, 0, ns:] = DUMMY_ROW
        Tv = T * v
        dyn = np.stack([Tv * cs, Tv * sn, T * om], axis=-1)             # [B, N, Nr, 3]
        g[:, 1:, :ns] = (X[:, 1:] - (X[:, :N] + dyn)).reshape(B, N, ns)
        gS[:, 1:, :ns] = (np.abs(X[:, 1:]) + np.abs(X[:, :N]) + np.abs(dyn)).reshape(B, N, ns)
        if M:
            a, b = np.array([p[0] for p in self.pairs]), np.array([p[1] for p in self.pairs])
            dx, dy = X[:, :N, a, 0] - X[:, :N, b, 0], X[:, :N, a, 1] - X[:, :N, b, 1]      # [B, N, M]
            g[:, 1:, ns:] = dx * dx + dy * dy
            gS[:, 1:, ns:] = g[:, 1:, ns:]
        out["g"] = (g.reshape(B, -1), np.abs(gS.reshape(B, -1)))
        # dg/dw at the pattern's slots
        rs = {"Tvs": Tv * sn, "mTvc": -T * v * cs, "mTc": -T * cs, "mTs": -T * sn}
        rs = {k: a.reshape(B, N * Nr) for k, a in rs.items()}
        if M:
            rs.update(p0=2 * dx, pm0=-2 * dx, p1=2 * dy, pm1=-2 * dy)
            for k in ("p0", "pm0", "p1", "pm1"):
                rs[k] = rs[k].reshape(B, N * M)
        jac = np.empty((B, d["nnzj"]), dtype=W.dtype)
        for key, (slots, at) in self.jac_kinds.items():
            jac[:, slots] = key[1] if isinstance(key, tuple) else rs[key][:, at]
        out["jac"] = (jac, np.abs(jac))
        if LAM is None:
            return out
        # hess(f + lam'g), lower triangle: the kernel sums 2 mu over the robot's pairs in order of the other robot
        L = LAM.reshape(B, N + 1, blk)[:, 1:]
        lx, ly = L[:, :, 0:ns:3].reshape(B, N, Nr), L[:, :, 1:ns:3].reshape(B, N, Nr)
        mu = L[:, :, ns:]
        sm2 = np.zeros((B, N, Nr), dtype=W.dtype)
        sm2S = np.zeros((B, N, Nr), dtype=W.dtype)
        pidx = {ab: q for q, ab in enumerate(self.pairs)}
        for i in range(Nr):
            for j in range(Nr):
                if j != i:
                    t = 2.0 * mu[:, :, pidx[(min(i, j), max(i, j))]]
                    sm2[:, :, i] = sm2[:, :, i] + t
                    sm2S[:, :, i] = sm2S[:, :, i] + np.abs(t)
        hv = {"xx": (2 * Qv[0] + sm2, 2 * abs(Qv[0]) + sm2S), "yy": (2 * Qv[1] + sm2, 2 * abs(Qv[1]) + sm2S),
              "tt": (2 * Qv[2] + Tv * (lx * cs + ly * sn), 2 * abs(Qv[2]) + np.abs(Tv) * (np.abs(lx * cs) + np.abs(ly * sn))),
              "vt": (T * (lx * sn - ly * cs), abs(T) * (np.abs(lx * sn) + np.abs(ly * cs)))}
        hv = {k: (a.reshape(B, N * Nr), s.reshape(B, N * Nr)) for k, (a, s) in hv.items()}
        if M:
            hv["mu"] = ((-2 * mu).reshape(B, N * M), np.abs(2 * mu).reshape(B, N * M))
        hess = np.empty((B, d["nnzh"]), dtype=W.dtype)
        hS = np.empty((B, d["nnzh"]), dtype=W.dtype)
        for key, (slots, at) in self.hess_kinds.items():
            if isinstance(key, tuple):
                hess[:, slots], hS[:, slots] = key[1], abs(key[1])
            else:
                hess[:, slots], hS[:, slots] = hv[key][0][:, at], hv[key][1][:, at]
        out["hess"] = (hess, hS)
        return out


def excess(dev, ref, S, k):
    """Largest |dev - ref| / (k eps S) over the entries: 0 where they are equal, inf where S = 0 and they differ or where
    either side is NaN.  <= 1 means within the bound."""
    dev, ref, S = (np.asarray(a, np.float64) for a in (dev, ref, S))
    diff = np.abs(dev - ref)
    tol = k * EPS * S
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(tol > 0, diff / np.where(tol > 0, tol, 1.0), np.where(diff == 0, 0.0, np.inf))
    r[~np.isfinite(diff)] = np.inf
    return float(r.max(initial=0.0))


EVAL_K = 8.0      # CUDA's double sin / cos (2 ulp), libm's (about 1 ulp) and FMA contraction


def record_excess(ref, out, k=EVAL_K):
    """{name: largest error / bound} of a device record `out` ({name: [B, ...] float64}) against EvalRef.eval's `ref`; the
    bound is k eps S per entry, and (n_terms + k) eps sum|terms| for f."""
    res = {}
    for name, val in out.items():
        if name == "f":
            f, S, nt = ref["f"]
            res[name] = excess(val, f, S, nt + k)
        else:
            res[name] = excess(val, ref[name][0], ref[name][1], k)
    return res


def shift(W, Nr, N):
    """nmpc_shift over a batch: X <- [X_1..X_N, X_{N-1}], U <- [U_1..U_{N-1}, U_{N-1}] (oracle/nlp_numpy.shift_warm_start)."""
    B, nX = W.shape[0], 3 * Nr * (N + 1)
    X, U = W[:, :nX].reshape(B, N + 1, 3 * Nr), W[:, nX:].reshape(B, N, 2 * Nr)
    return np.concatenate([np.concatenate([X[:, 1:], X[:, N - 1:N]], axis=1).reshape(B, -1),
                           np.concatenate([U[:, 1:], U[:, -1:]], axis=1).reshape(B, -1)], axis=1)


def plant(state, xopt, Nr, N, T, sin=np.sin, cos=np.cos):
    """nmpc_plant over a batch: (x, y, th) + T (v cos th, v sin th, om) with U_0 of xopt.  Returns (next state, S) with
    S = |x| + |T v cos th| (|y| + |T v sin th|, |th| + |T om|) per component."""
    B, nX = state.shape[0], 3 * Nr * (N + 1)
    s = state.reshape(B, Nr, 3)
    u = xopt[:, nX:nX + 2 * Nr].reshape(B, Nr, 2)
    th = s[..., 2]
    inc = np.stack([T * u[..., 0] * cos(th), T * u[..., 0] * sin(th), T * u[..., 1]], axis=-1)
    return (s + inc).reshape(B, -1), (np.abs(s) + np.abs(inc)).reshape(B, -1)
