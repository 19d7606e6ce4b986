"""Host side of the hot path: the nlpsol-compatible call surface and the batched device API.

Mirrors what the reference does around its solver call
(AllScripts/centralized_six_robots_implementation.py):
    solver = nlpsol('solver', 'ipopt', nlp_prob, opts)        :345-346
    sol = solver(x0=..., p=..., lbx=..., ubx=..., lbg=..., ubg=...)   :432
    sol['x'][a:b] ... .full()                                  :436,440,460
so that the scenario loops (:416-510) run unchanged on top of the CUDA library.  CasADi is not a
dependency: the factory takes a problem descriptor in place of the symbolic dict (SURVEY.md 8b).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _cabi
from ._cabi import NSTATS, NTRACE, Desc, NmpcError, check, default_opts, default_tuning, lib


# ----------------------------------------------------------------------------------------------
# the few CasADi names the reference's loop bodies use on numeric data (SURVEY.md App. E)
# ----------------------------------------------------------------------------------------------
class DM:
    """Dense numeric matrix with CasADi's column-major semantics: [a:b] slicing on the flattened
    column-major vector, .full() -> ndarray, usable wherever NumPy expects an array."""

    def __init__(self, a):
        a = np.asarray(a.full() if isinstance(a, DM) else a, dtype=float)
        self._a = a.reshape(-1, 1) if a.ndim < 2 else a

    def full(self):
        return self._a.copy()

    @property
    def shape(self):
        return self._a.shape

    def numel(self):
        return self._a.size

    def __array__(self, dtype=None, copy=None):
        return self._a.astype(dtype) if dtype is not None else self._a

    def __len__(self):
        return self._a.shape[0]

    def __getitem__(self, idx):
        if isinstance(idx, tuple):
            return DM(np.atleast_2d(self._a[idx]))
        flat = self._a.reshape(-1, order="F")
        return DM(np.atleast_1d(flat[idx]).reshape(-1, 1))

    def __float__(self):
        return float(self._a.reshape(-1)[0])

    def __repr__(self):
        return "DM(%r)" % (self._a,)


def _num(a):
    return np.asarray(a.full() if isinstance(a, DM) else a, dtype=float)


def reshape(a, *shape):
    """CasADi reshape: column-major."""
    if len(shape) == 1:
        shape = tuple(shape[0])
    return DM(np.reshape(np.atleast_2d(_num(a)), (int(shape[0]), int(shape[1])), order="F"))


def repmat(a, n, m=1):
    return DM(np.tile(np.atleast_2d(_num(a)), (int(n), int(m))))


def vertcat(*args):
    return DM(np.concatenate([np.atleast_2d(_num(a)).reshape(-1, np.atleast_2d(_num(a)).shape[-1]) if np.ndim(_num(a)) > 1
                              else _num(a).reshape(-1, 1) for a in args], axis=0))


def horzcat(*args):
    return DM(np.concatenate([np.atleast_2d(_num(a)) for a in args], axis=1))


def _flat(a, size, name):
    """Accept row or column vectors, scalars (broadcast) and DM; flatten column-major."""
    v = _num(a)
    if v.size == 1:
        return np.full(size, float(v.reshape(-1)[0]))
    v = v.reshape(-1, order="F")
    if v.size != size:
        raise ValueError("%s has %d entries, expected %d" % (name, v.size, size))
    return np.ascontiguousarray(v, dtype=np.float64)


# ----------------------------------------------------------------------------------------------
class Problem:
    """Handle on the CUDA library for one (Nr, N, T, Q, R) problem family."""

    def __init__(self, Nr, N, T, Q=(1.0, 5.0, 0.1), R=(0.5, 0.05), obstacles=None, tuning=None, moving_obstacles=None,
                 tracking=False, tracking_obstacles=None, **opts):
        """obstacles: optional [n_obs, 3] array of static circular obstacles (centre x, y, clearance = rob_dim + r_obs): the
        reference's obstacle-avoidance family (first_scenario_mpc_obstacle_avoidance.py:96-152), see nmpc_create_obstacles.
        moving_obstacles: n_obs instead of `obstacles` -> the same family with the obstacles in p, one [n_obs, 3] table per
        instance and stage (p = [x0bar; xs; O[N][n_obs][3]], see nmpc_create_moving_obstacles and params()).
        tracking: True -> the centralized family tracking a per-instance, per-stage state and control reference instead of one
        goal (p = [x0bar; Z[N][5Nr]], Z[k] = [xr_k; ur_k], see nmpc_create_tracking and params()); no obstacles.
        tracking_obstacles: n_obs -> both: the moving-obstacle family tracking a per-stage reference, p = [x0bar; Z[N][5Nr];
        O[N][n_obs][3]] (see nmpc_create_tracking_obstacles and params()); exclusive with the three keywords above.  The
        handle has tracking = moving = True.
        tuning: optional dict of nmpc_tuning fields (convoy, ctas_per_sm, force_block_path, thread_min_batch)."""
        if obstacles is not None and moving_obstacles is not None:
            raise ValueError("obstacles= and moving_obstacles= are mutually exclusive")
        if tracking and (obstacles is not None or moving_obstacles is not None):
            raise ValueError("tracking=True cannot be combined with obstacles= or moving_obstacles=")
        if tracking_obstacles is not None and (tracking or obstacles is not None or moving_obstacles is not None):
            raise ValueError("tracking_obstacles= cannot be combined with tracking=, obstacles= or moving_obstacles=")
        self.L = lib()
        self.desc = Desc(int(Nr), int(N), float(T), (C.c_double * 3)(*[float(q) for q in Q]),
                         (C.c_double * 2)(*[float(r) for r in R]))
        self.opts = default_opts(**opts)
        self.h = C.c_void_p()
        self.obstacles = None if obstacles is None else np.ascontiguousarray(np.asarray(obstacles, dtype=np.float64).reshape(-1, 3))
        self.tuning = default_tuning(**(tuning or {}))
        self.moving = moving_obstacles is not None or tracking_obstacles is not None
        self.tracking = bool(tracking) or tracking_obstacles is not None
        if tracking_obstacles is not None:
            check(self.L.nmpc_create_tracking_obstacles(C.byref(self.desc), C.byref(self.opts), C.byref(self.tuning),
                                                        int(tracking_obstacles), C.byref(self.h)))
            self.nobs = int(tracking_obstacles)
        elif self.tracking:
            check(self.L.nmpc_create_tracking(C.byref(self.desc), C.byref(self.opts), C.byref(self.tuning), C.byref(self.h)))
            self.nobs = 0
        elif self.moving:
            check(self.L.nmpc_create_moving_obstacles(C.byref(self.desc), C.byref(self.opts), C.byref(self.tuning),
                                                      int(moving_obstacles), C.byref(self.h)))
            self.nobs = int(moving_obstacles)
        else:
            check(self.L.nmpc_create_tuned(C.byref(self.desc), C.byref(self.opts), C.byref(self.tuning),
                                           0 if self.obstacles is None else int(self.obstacles.shape[0]),
                                           None if self.obstacles is None else self.obstacles.ctypes.data, C.byref(self.h)))
            self.nobs = 0 if self.obstacles is None else int(self.obstacles.shape[0])
        self.Nr, self.N, self.T = int(Nr), int(N), float(T)
        self.ns, self.nc = 3 * self.Nr, 2 * self.Nr
        self.M = self.Nr * (self.Nr - 1) // 2
        self.n, self.mg, self.np_ = self.L.nmpc_n(self.h), self.L.nmpc_mg(self.h), self.L.nmpc_np(self.h)
        self.nnz_jac, self.nnz_hess = self.L.nmpc_nnz_jac(self.h), self.L.nmpc_nnz_hess(self.h)
        self._ws = None

    def __del__(self):
        try:
            if self.h:
                self.L.nmpc_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # reference bounds (centralized_six_robots_implementation.py:349-352)
    def bounds(self, dmin, v_max, w_max, xy_box=10.0):
        inf = np.inf
        lbx = np.concatenate([np.tile([-xy_box, -xy_box, -inf], self.Nr * (self.N + 1)),
                              np.tile([-v_max, -w_max], self.Nr * self.N)])
        ubx = -lbx
        lbg = np.tile(np.concatenate([np.zeros(self.ns), np.full(self.M, dmin * dmin)]), self.N + 1)
        ubg = np.tile(np.concatenate([np.zeros(self.ns), np.full(self.M, inf)]), self.N + 1)
        return lbx, ubx, lbg, ubg

    def bounds_obstacles(self, margin, v_max, w_max, dmin=0.0, xy_box=10.0, th_box=2.0 * np.pi):
        """Bounds of the obstacle-avoidance scripts (first_scenario_mpc_obstacle_avoidance.py:150-152): theta boxed to +-2 pi,
        equality rows 0, obstacle rows >= margin (0.05 there, 0.1 in the third scenario), pair rows (Nr > 1) >= dmin^2."""
        inf = np.inf
        lbx = np.concatenate([np.tile([-xy_box, -xy_box, -th_box], self.Nr * (self.N + 1)),
                              np.tile([-v_max, -w_max], self.Nr * self.N)])
        ubx = -lbx
        blk_lo = np.concatenate([np.zeros(self.ns), np.full(self.M, dmin * dmin), np.full(self.Nr * self.nobs, margin)])
        blk_hi = np.concatenate([np.zeros(self.ns), np.full(self.M + self.Nr * self.nobs, inf)])
        lbg = np.concatenate([np.zeros(self.ns), np.tile(blk_lo, self.N)])
        ubg = np.concatenate([np.zeros(self.ns), np.tile(blk_hi, self.N)])
        return lbx, ubx, lbg, ubg

    def cold_start(self, x0):
        """X_k = x0 for all k, U = 0 (:398-400,423)."""
        x0 = np.asarray(x0, float)
        if x0.ndim == 1:
            return np.concatenate([np.tile(x0, self.N + 1), np.zeros(self.nc * self.N)])
        return np.concatenate([np.tile(x0, (1, self.N + 1)), np.zeros((x0.shape[0], self.nc * self.N))], axis=1)

    def params(self, x0bar, xs, obstacles=None, uref=None):
        """p [B, np] from x0bar [B, 3Nr], xs [B, 3Nr] and, for moving_obstacles, obstacles [B, N, n_obs, 3] (ox, oy, clearance of
        every obstacle at every stage).  For tracking: xs is the state reference [B, N, 3Nr] (or [B, 3Nr], the same at every
        stage) and uref the control reference [B, N, 2Nr] (default zeros); with tracking_obstacles also obstacles as above.
        NumPy arrays give a NumPy array, CUDA tensors a contiguous float64 tensor on their device."""
        B = x0bar.shape[0]
        if getattr(self, "tracking", False):
            return self._tracking_params(x0bar, xs, uref, obstacles)
        if uref is not None:
            raise ValueError("uref goes into p only for Problem(tracking=True)")
        if tuple(x0bar.shape) != (B, self.ns) or tuple(xs.shape) != (B, self.ns):
            raise ValueError("x0bar and xs must be [B, %d]" % self.ns)
        parts = [x0bar, xs]
        if self.moving:
            if obstacles is None or tuple(obstacles.shape) != (B, self.N, self.nobs, 3):
                raise ValueError("obstacles must be [B, N, n_obs, 3] = [%d, %d, %d, 3]" % (B, self.N, self.nobs))
            parts.append(obstacles.reshape(B, -1))
        elif obstacles is not None:
            raise ValueError("obstacles go into p only for Problem(moving_obstacles=n_obs)")
        if isinstance(x0bar, np.ndarray):
            return np.ascontiguousarray(np.concatenate([np.asarray(a, np.float64) for a in parts], axis=1))
        torch = self._torch()
        return torch.cat([a.to(torch.float64) for a in parts], dim=1).contiguous()

    def _tracking_params(self, x0bar, xs, uref, obstacles):
        B, N = x0bar.shape[0], self.N
        if self.moving:     # tracking_obstacles: O[N][n_obs][3] after Z
            if obstacles is None or tuple(obstacles.shape) != (B, N, self.nobs, 3):
                raise ValueError("obstacles must be [B, N, n_obs, 3] = [%d, %d, %d, 3]" % (B, N, self.nobs))
        elif obstacles is not None:
            raise ValueError("obstacles go into p only for Problem(moving_obstacles=n_obs)")
        if tuple(x0bar.shape) != (B, self.ns) or tuple(xs.shape) not in ((B, self.ns), (B, N, self.ns)):
            raise ValueError("x0bar must be [B, %d] and xs [B, N, %d] or [B, %d]" % (self.ns, self.ns, self.ns))
        if uref is not None and tuple(uref.shape) != (B, N, self.nc):
            raise ValueError("uref must be [B, N, 2Nr] = [%d, %d, %d]" % (B, N, self.nc))
        if isinstance(x0bar, np.ndarray):
            xr = np.broadcast_to(np.asarray(xs, np.float64).reshape(B, -1, self.ns), (B, N, self.ns))
            ur = np.zeros((B, N, self.nc)) if uref is None else np.asarray(uref, np.float64)
            Z = np.concatenate([xr, ur], axis=2).reshape(B, -1)
            parts = [np.asarray(x0bar, np.float64), Z]
            if obstacles is not None:
                parts.append(np.asarray(obstacles, np.float64).reshape(B, -1))
            return np.ascontiguousarray(np.concatenate(parts, axis=1))
        torch = self._torch()
        xr = xs.to(torch.float64).reshape(B, -1, self.ns).expand(B, N, self.ns)
        ur = (torch.zeros((B, N, self.nc), dtype=torch.float64, device=xs.device) if uref is None else uref.to(torch.float64))
        parts = [x0bar.to(torch.float64), torch.cat([xr, ur], dim=2).reshape(B, -1)]
        if obstacles is not None:
            parts.append(obstacles.to(torch.float64).reshape(B, -1))
        return torch.cat(parts, dim=1).contiguous()

    def launch_count(self):
        return int(self.L.nmpc_launch_count(self.h))

    def jac_pattern(self):
        cp, ri = np.zeros(self.n + 1, np.int32), np.zeros(self.nnz_jac, np.int32)
        check(self.L.nmpc_jac_pattern(self.h, cp.ctypes.data, ri.ctypes.data))
        return cp, ri

    def hess_pattern(self):
        cp, ri = np.zeros(self.n + 1, np.int32), np.zeros(self.nnz_hess, np.int32)
        check(self.L.nmpc_hess_pattern(self.h, cp.ctypes.data, ri.ctypes.data))
        return cp, ri

    # ---- host-buffer path (what a CasADi-style caller has) -------------------------------------
    def solve_host(self, x0, p, lbx, ubx, lbg, ubg, want=("f", "g", "lam_x", "lam_g", "stats"), out=None):
        f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        x0, p = np.atleast_2d(f64(x0)), np.atleast_2d(f64(p))
        lbx, ubx, lbg, ubg = f64(lbx), f64(ubx), f64(lbg), f64(ubg)
        B = x0.shape[0]
        if getattr(self, "_order", None) is not None and self._order.numel() != B:
            raise ValueError("the scheduling order set with set_order() has %d entries, the batch has %d" % (self._order.numel(), B))
        if x0.shape[1] != self.n or p.shape != (B, self.np_):
            raise ValueError("x0 must be [B,%d] and p [B,%d]" % (self.n, self.np_))
        batched = 1 if lbx.ndim == 2 else 0
        for a, m, nm in ((lbx, self.n, "lbx"), (ubx, self.n, "ubx"), (lbg, self.mg, "lbg"), (ubg, self.mg, "ubg")):
            if a.shape != ((B, m) if batched else (m,)):
                raise ValueError("%s has shape %s" % (nm, a.shape))
        o = out if out is not None else {}
        o.setdefault("x", np.empty((B, self.n)))
        for k, shp in (("f", (B,)), ("g", (B, self.mg)), ("lam_x", (B, self.n)), ("lam_g", (B, self.mg)), ("stats", (B, NSTATS))):
            if k in want:
                o.setdefault(k, np.empty(shp))
        o.setdefault("status", np.empty(B, np.int32))
        o.setdefault("iters", np.empty(B, np.int32))
        ptr = lambda k: o[k].ctypes.data if k in o else None
        check(self.L.nmpc_solve_host(self.h, B, x0.ctypes.data, p.ctypes.data, lbx.ctypes.data, ubx.ctypes.data,
                                     lbg.ctypes.data, ubg.ctypes.data, batched, ptr("x"), ptr("f"), ptr("g"),
                                     ptr("lam_x"), ptr("lam_g"), ptr("status"), ptr("iters"), ptr("stats")))
        return o

    # ---- device path: torch CUDA tensors, zero-copy, asynchronous on the current stream --------
    def _torch(self):
        import torch
        if not torch.cuda.is_available():
            raise NmpcError("no CUDA device: the batched path has no CPU fallback")
        return torch

    def workspace(self, B, batched_bounds=False, device=None):
        torch = self._torch()
        need = (self.L.nmpc_workspace_bytes_batched_bounds if batched_bounds else self.L.nmpc_workspace_bytes)(self.h, int(B))
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        if self._ws is None or self._ws.numel() < need or self._ws.device != device:
            self._ws = torch.empty(int(need), dtype=torch.uint8, device=device)
        return self._ws

    def _stream(self, device):
        """Raw stream handle of torch's current stream ON THE TENSORS' DEVICE (the handle checks the device itself)."""
        return self._torch().cuda.current_stream(device).cuda_stream

    def solve(self, x0, p, lbx, ubx, lbg, ubg, want=("f", "g", "lam_x", "lam_g", "stats"), out=None, trace=0):
        """x0 [B,n], p [B,6Nr], bounds [n]/[mg] or [B,.]: float64 CUDA tensors.  Returns CUDA tensors."""
        torch = self._torch()
        B = x0.shape[0]
        for t in (x0, p, lbx, ubx, lbg, ubg):
            if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
                raise ValueError("inputs must be contiguous float64 CUDA tensors")
        if getattr(self, "_order", None) is not None and self._order.numel() != B:
            raise ValueError("the scheduling order set with set_order() has %d entries, the batch has %d" % (self._order.numel(), B))
        batched = 1 if lbx.dim() == 2 else 0
        dev = x0.device
        if any(t.device != dev for t in (p, lbx, ubx, lbg, ubg)):
            raise ValueError("all inputs must live on the same CUDA device")
        if self.np_ > 0 and tuple(p.shape) != (B, self.np_):
            raise ValueError("p must be [B, %d], got %s" % (self.np_, tuple(p.shape)))
        ws = self.workspace(B, bool(batched), dev)
        o = out if out is not None else {}
        o.setdefault("x", torch.empty((B, self.n), dtype=torch.float64, device=dev))
        for k, shp in (("f", (B,)), ("g", (B, self.mg)), ("lam_x", (B, self.n)), ("lam_g", (B, self.mg)), ("stats", (B, NSTATS))):
            if k in want:
                o.setdefault(k, torch.empty(shp, dtype=torch.float64, device=dev))
        o.setdefault("status", torch.empty(B, dtype=torch.int32, device=dev))
        o.setdefault("iters", torch.empty(B, dtype=torch.int32, device=dev))
        ptr = lambda k: o[k].data_ptr() if k in o else None
        stream = self._stream(dev)
        args = [self.h, B, x0.data_ptr(), p.data_ptr(), lbx.data_ptr(), ubx.data_ptr(), lbg.data_ptr(), ubg.data_ptr(), batched,
                ptr("x"), ptr("f"), ptr("g"), ptr("lam_x"), ptr("lam_g"), ptr("status"), ptr("iters"), ptr("stats")]
        if trace:
            o["trace"] = torch.zeros((B, int(trace), NTRACE), dtype=torch.float64, device=dev)
            check(self.L.nmpc_solve_trace(*args, o["trace"].data_ptr(), int(trace), ws.data_ptr(), ws.numel(), stream))
        else:
            check(self.L.nmpc_solve(*args, ws.data_ptr(), ws.numel(), stream))
        return o

    # ---- parametric sensitivities of returned solutions (nmpc_solution_vjp / nmpc_solution_jvp) ---------------------------
    def _sensitivity(self, fn, out, p, lbx, ubx, lbg, ubg, seed, seed_cols, out_cols):
        torch = self._torch()
        x, lam_x, lam_g = out["x"], out["lam_x"], out["lam_g"]
        B, dev = x.shape[0], x.device
        for t in (x, lam_x, lam_g, p, lbx, ubx, lbg, ubg, seed):
            if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and t.device == dev):
                raise ValueError("inputs must be contiguous float64 CUDA tensors on one device")
        if tuple(seed.shape) != (B, seed_cols) or tuple(p.shape) != (B, self.np_):
            raise ValueError("p must be [B, %d] and the seed [B, %d]" % (self.np_, seed_cols))
        batched = 1 if lbx.dim() == 2 else 0
        need = int(self.L.nmpc_sensitivity_workspace_bytes(self.h, B, batched))
        if getattr(self, "_sws", None) is None or self._sws.numel() < need or self._sws.device != dev:
            self._sws = torch.empty(max(need, 1), dtype=torch.uint8, device=dev)
        res = torch.empty((B, out_cols), dtype=torch.float64, device=dev)
        st = torch.empty(B, dtype=torch.int32, device=dev)
        check(fn(self.h, B, x.data_ptr(), lam_x.data_ptr(), lam_g.data_ptr(), p.data_ptr(), lbx.data_ptr(), ubx.data_ptr(),
                 lbg.data_ptr(), ubg.data_ptr(), batched, seed.data_ptr(), res.data_ptr(), st.data_ptr(), self._sws.data_ptr(), need,
                 self._stream(dev)))
        return res, st

    def solution_vjp(self, out, p, lbx, ubx, lbg, ubg, x_bar):
        """Reverse-mode derivative of the solution: p_bar [B, np] = x_bar' dx*/dp for x_bar [B, n], at the solutions `out` (the
        dict solve() returned: x, lam_x, lam_g) of the solve with this p and these bounds.  Returns (p_bar, sens_status):
        status 0 ok, 1 wrong inertia at the point (p_bar is NaN there), < 0 bounds rejected.  See nmpc_solution_vjp."""
        return self._sensitivity(self.L.nmpc_solution_vjp, out, p, lbx, ubx, lbg, ubg, x_bar, self.n, self.np_)

    def solution_jvp(self, out, p, lbx, ubx, lbg, ubg, p_dot):
        """Forward-mode derivative of the solution: x_dot [B, n] = dx*/dp p_dot for p_dot [B, np]; (x_dot, sens_status) as in
        solution_vjp.  x + x_dot is the first-order prediction of the solution at p + p_dot (the sensitivity correction of an
        advanced-step controller)."""
        return self._sensitivity(self.L.nmpc_solution_jvp, out, p, lbx, ubx, lbg, ubg, p_dot, self.np_, self.n)

    def solve_differentiable(self, x0, p, lbx, ubx, lbg, ubg):
        """solve() as a torch.autograd function of p: returns x [B, n]; x.backward / torch.autograd.grad give the gradient with
        respect to p through nmpc_solution_vjp at the returned solutions.  x0 and the bounds get no gradient (x* does not depend
        on the start point; derivatives with respect to the bounds are not provided).  An instance whose solve did not converge
        gets the derivative of its returned point all the same; one with the wrong inertia there gets NaN."""
        return _solve_function().apply(self, x0, p, lbx, ubx, lbg, ubg)

    def set_order(self, order=None):
        """Scheduling hint (nmpc_set_order): int32 CUDA tensor [B], a permutation of the instances, longest expected solve
        first; None restores index order.  The tensor is kept alive by the handle."""
        if order is not None:
            torch = self._torch()
            if not (order.is_cuda and order.dtype == torch.int32 and order.is_contiguous()):
                raise ValueError("order must be a contiguous int32 CUDA tensor")
        self._order = order
        check(self.L.nmpc_set_order(self.h, None if order is None else order.data_ptr(), 0 if order is None else int(order.numel())))

    def order_from_iters(self, iters):
        """Longest-first order from the iteration counts of the previous MPC step (the closed-loop predictor)."""
        torch = self._torch()
        return torch.argsort(iters, descending=True, stable=True).to(torch.int32).contiguous()

    def shift(self, x_prev, out=None):
        torch = self._torch()
        out = torch.empty_like(x_prev) if out is None else out
        check(self.L.nmpc_shift(self.h, x_prev.shape[0], x_prev.data_ptr(), out.data_ptr(), self._stream(x_prev.device)))
        return out

    def plant(self, state, x_opt, out=None):
        torch = self._torch()
        out = torch.empty_like(state) if out is None else out
        check(self.L.nmpc_plant(self.h, state.shape[0], state.data_ptr(), x_opt.data_ptr(), out.data_ptr(), self._stream(state.device)))
        return out

    def eval(self, w, p, lam_g=None, want=("f", "grad", "g", "jac", "hess")):
        torch = self._torch()
        B, dev = w.shape[0], w.device
        o = {}
        shapes = dict(f=(B,), grad=(B, self.n), g=(B, self.mg), jac=(B, self.nnz_jac), hess=(B, self.nnz_hess))
        for k in want:
            if k == "hess" and lam_g is None:
                continue
            o[k] = torch.empty(shapes[k], dtype=torch.float64, device=dev)
        ptr = lambda k: o[k].data_ptr() if k in o else None
        check(self.L.nmpc_eval(self.h, B, w.data_ptr(), p.data_ptr(), lam_g.data_ptr() if lam_g is not None else None,
                               ptr("f"), ptr("grad"), ptr("g"), ptr("jac"), ptr("hess"), self._stream(dev)))
        return o


_SOLVE_FUNCTION = None


def _solve_function():
    """The torch.autograd.Function behind Problem.solve_differentiable (built on first use: torch is imported lazily)."""
    global _SOLVE_FUNCTION
    if _SOLVE_FUNCTION is None:
        import torch

        class SolveFunction(torch.autograd.Function):
            @staticmethod
            def forward(ctx, prob, x0, p, lbx, ubx, lbg, ubg):
                out = prob.solve(x0, p.detach(), lbx, ubx, lbg, ubg, want=("lam_x", "lam_g"))
                ctx.prob = prob
                ctx.save_for_backward(p.detach(), lbx, ubx, lbg, ubg, out["x"], out["lam_x"], out["lam_g"])
                return out["x"]

            @staticmethod
            @torch.autograd.function.once_differentiable
            def backward(ctx, x_bar):
                p, lbx, ubx, lbg, ubg, x, lam_x, lam_g = ctx.saved_tensors
                p_bar, _ = ctx.prob.solution_vjp(dict(x=x, lam_x=lam_x, lam_g=lam_g), p, lbx, ubx, lbg, ubg,
                                                 x_bar.to(torch.float64).contiguous())
                return None, None, p_bar, None, None, None, None

        _SOLVE_FUNCTION = SolveFunction
    return _SOLVE_FUNCTION


def closed_loop(prob, P, lbx, ubx, lbg, ubg, steps, tol=1e-1, dmin=None, obstacles=None, reference=None):
    """Batched closed-loop driver, device resident (SURVEY.md 8f-1): the reference's loop body
    (centralized_six_robots_implementation.py:416-465 with the Euler plant of casadi_test.py:17-26) for B
    independent instances at once.  Per step: solve -> apply u_0 through the plant -> reference shift as the next
    guess; instances whose ||x - xs|| <= tol stop moving (the loop guard at :416).  Returns a dict of CUDA tensors:
    traj [steps+1,B,3Nr], u [steps,B,2Nr], status [steps,B], iters [steps,B], active [steps,B], min_dist [B].
    obstacles (Problem(moving_obstacles=n_obs) only): CUDA float64 [steps+N, B, n_obs, 3], the obstacles' positions and
    clearances over time; step t solves with the window t..t+N-1 in p (P then needs only its first 6Nr columns), and the
    result gains min_clearance [B] = min over time, robots and obstacles of rho - clearance between the plant state and the
    obstacles at the same time.
    reference (required by, and only for, Problem(tracking=True)): CUDA float64 [steps+N, B, 5Nr], rows [xr_t; ur_t] of the
    reference over time; step t solves with rows t..t+N-1 as Z in p (P then needs only its first 3Nr columns, x0bar), there is
    no stop test (every instance is active at every step), and the result gains track_err [steps+1, B] = the largest xy distance
    over robots between the plant state and the reference state at the same time.
    Problem(tracking_obstacles=n_obs) requires both: step t solves with Z = reference rows t..t+N-1 and O = obstacle tables
    t..t+N-1 (P then needs only x0bar), without a stop test, and the result carries both track_err and min_clearance."""
    torch = prob._torch()
    B, ns, nc, N = P.shape[0], prob.ns, prob.nc, prob.N
    tracking = getattr(prob, "tracking", False)
    both = tracking and getattr(prob, "moving", False)      # Problem(tracking_obstacles=n_obs)
    if both and (reference is None or obstacles is None):
        raise ValueError("a Problem(tracking_obstacles=n_obs) needs both reference= and obstacles=")
    if tracking != (reference is not None):
        raise ValueError("reference= is required by, and only accepted for, a Problem(tracking=True)")
    if both:
        if not (reference.is_cuda and reference.dtype == torch.float64) or tuple(reference.shape) != (steps + N, B, ns + nc):
            raise ValueError("reference must be a float64 CUDA tensor [steps + N, B, 5Nr] = [%d, %d, %d]" % (steps + N, B, ns + nc))
        if not (obstacles.is_cuda and obstacles.dtype == torch.float64) or tuple(obstacles.shape) != (steps + N, B, prob.nobs, 3):
            raise ValueError("obstacles must be a float64 CUDA tensor [steps + N, B, n_obs, 3] = [%d, %d, %d, 3]"
                             % (steps + N, B, prob.nobs))
        p = torch.empty((B, prob.np_), dtype=torch.float64, device=P.device)
        p[:, :ns] = P[:, :ns]
    elif tracking:
        if not (reference.is_cuda and reference.dtype == torch.float64) or tuple(reference.shape) != (steps + N, B, ns + nc):
            raise ValueError("reference must be a float64 CUDA tensor [steps + N, B, 5Nr] = [%d, %d, %d]" % (steps + N, B, ns + nc))
        p = torch.cat([P[:, :ns], torch.empty((B, N * (ns + nc)), dtype=torch.float64, device=P.device)], dim=1)
    elif obstacles is not None:
        if not getattr(prob, "moving", False):
            raise ValueError("obstacles= needs a Problem(moving_obstacles=n_obs)")
        if not (obstacles.is_cuda and obstacles.dtype == torch.float64) or tuple(obstacles.shape) != (steps + N, B, prob.nobs, 3):
            raise ValueError("obstacles must be a float64 CUDA tensor [steps + N, B, n_obs, 3] = [%d, %d, %d, 3]"
                             % (steps + N, B, prob.nobs))
        p = torch.cat([P[:, :2 * ns], torch.empty((B, 3 * N * prob.nobs), dtype=torch.float64, device=P.device)], dim=1)
    else:
        p = P.clone()
    x0 = torch.cat([p[:, :ns].repeat(1, N + 1), torch.zeros((B, nc * N), dtype=torch.float64, device=P.device)], dim=1).contiguous()
    traj = torch.empty((steps + 1, B, ns), dtype=torch.float64, device=P.device)
    us = torch.zeros((steps, B, nc), dtype=torch.float64, device=P.device)
    st = torch.zeros((steps, B), dtype=torch.int32, device=P.device)
    its = torch.zeros((steps, B), dtype=torch.int32, device=P.device)
    act = torch.zeros((steps, B), dtype=torch.bool, device=P.device)
    traj[0] = p[:, :ns]
    out = {}
    for t in range(steps):
        if t == 0:
            prob.set_order(None)
        if both:
            p[:, ns:ns + N * (ns + nc)] = reference[t:t + N].permute(1, 0, 2).reshape(B, -1)
            p[:, ns + N * (ns + nc):] = obstacles[t:t + N].permute(1, 0, 2, 3).reshape(B, -1)
        elif obstacles is not None:
            p[:, 2 * ns:] = obstacles[t:t + N].permute(1, 0, 2, 3).reshape(B, -1)
        if tracking:
            if not both:
                p[:, ns:] = reference[t:t + N].permute(1, 0, 2).reshape(B, -1)
            active = torch.ones(B, dtype=torch.bool, device=P.device)
        else:
            active = (p[:, :ns] - p[:, ns:2 * ns]).norm(dim=1) > tol
        act[t] = active
        prob.solve(x0, p, lbx, ubx, lbg, ubg, want=(), out=out)
        u0 = out["x"][:, ns * (N + 1):ns * (N + 1) + nc]
        nxt = prob.plant(p[:, :ns].contiguous(), out["x"])
        p[:, :ns] = torch.where(active[:, None], nxt, p[:, :ns])
        us[t] = torch.where(active[:, None], u0, torch.zeros_like(u0))
        st[t], its[t] = out["status"], out["iters"]
        prob.set_order(prob.order_from_iters(out["iters"]))      # longest solves first in the next step
        x0 = prob.shift(out["x"])
        traj[t + 1] = p[:, :ns]
    prob.set_order(None)
    res = dict(traj=traj, u=us, status=st, iters=its, active=act)
    if prob.Nr > 1:
        pos = traj.reshape(steps + 1, B, prob.Nr, 3)[..., :2]
        d = (pos[:, :, :, None, :] - pos[:, :, None, :, :]).norm(dim=-1)
        d = d + torch.eye(prob.Nr, device=P.device, dtype=torch.float64)[None, None] * 1e9
        res["min_dist"] = d.amin(dim=(0, 2, 3))
    if obstacles is not None:
        pos = traj.reshape(steps + 1, B, prob.Nr, 3)[..., :2]
        ob = obstacles[:steps + 1]
        rho = (pos[:, :, :, None, :] - ob[:, :, None, :, :2]).norm(dim=-1)
        res["min_clearance"] = (rho - ob[:, :, None, :, 2]).amin(dim=(0, 2, 3))
    if tracking:
        pos = traj.reshape(steps + 1, B, prob.Nr, 3)[..., :2]
        ref = reference[:steps + 1, :, :ns].reshape(steps + 1, B, prob.Nr, 3)[..., :2]
        res["track_err"] = (pos - ref).norm(dim=-1).amax(dim=2)
    return res


class SmallOcp(Problem):
    """Small generic OCP, one GPU thread per instance (nmpc_create_ocp).  model 'van_der_pol' is the direct-multiple-shooting
    demo of mpc_pose_control_casadi.py:22-114: interleaved decision vector [X_0, U_0, ..., X_N] (n = 3N + 2), g = F(X_k, U_k) -
    X_{k+1} (mg = 2N), initial state fixed through its bounds, no parameter vector."""
    MODELS = {"van_der_pol": 1}

    def __init__(self, model="van_der_pol", N=20, T=10.0, rk_steps=4, **opts):
        self.L = lib()
        self.opts = default_opts(**({"max_iter": 3000} | opts))      # the demo sets no options: IPOPT's default max_iter
        self.h = C.c_void_p()
        check(self.L.nmpc_create_ocp(self.MODELS[model], int(N), float(T), int(rk_steps), C.byref(self.opts), C.byref(self.h)))
        self.model, self.Nr, self.N, self.T, self.rk_steps = model, 0, int(N), float(T), int(rk_steps)
        self.ns, self.nc, self.M, self.nobs, self.obstacles = 2, 1, 0, 0, None
        self.n, self.mg, self.np_ = self.L.nmpc_n(self.h), self.L.nmpc_mg(self.h), 0
        self.nnz_jac = self.nnz_hess = 0
        self._ws = None

    def demo_arrays(self):
        """w0, lbw, ubw, lbg, ubg exactly as the demo assembles them (mpc_pose_control_casadi.py:77-106)."""
        inf = np.inf
        w0, lbw, ubw = [0.0, 1.0], [0.0, 1.0], [0.0, 1.0]
        for _ in range(self.N):
            w0 += [0.0, 0.0, 0.0]; lbw += [-1.0, -0.25, -inf]; ubw += [1.0, inf, inf]
        return np.array(w0), np.array(lbw), np.array(ubw), np.zeros(self.mg), np.zeros(self.mg)

    def solve_host(self, x0, lbx, ubx, lbg, ubg, want=("f", "g", "lam_x", "lam_g", "stats"), out=None):
        x0 = np.atleast_2d(np.ascontiguousarray(x0, dtype=np.float64))
        return Problem.solve_host(self, x0, np.zeros((x0.shape[0], 0)), lbx, ubx, lbg, ubg, want=want, out=out)


class NlpSolver:
    """What nlpsol(...) returns: callable with the reference's keyword arguments (:432)."""

    def __init__(self, name, problem):
        self.name, self.problem = name, problem
        self._stats = {}

    def __call__(self, x0=0.0, p=None, lbx=-np.inf, ubx=np.inf, lbg=-np.inf, ubg=np.inf, lam_x0=None, lam_g0=None):
        P = self.problem
        if P.np_ == 0:      # parameter-free problem (the Van der Pol demo calls solver(x0=, lbx=, ubx=, lbg=, ubg=), :113)
            o = P.solve_host(_flat(x0, P.n, "x0")[None], _flat(lbx, P.n, "lbx"), _flat(ubx, P.n, "ubx"), _flat(lbg, P.mg, "lbg"),
                             _flat(ubg, P.mg, "ubg"))
        else:
            if p is None:
                raise ValueError("p = [x0; xs] is required")
            o = P.solve_host(_flat(x0, P.n, "x0")[None], _flat(p, P.np_, "p")[None], _flat(lbx, P.n, "lbx"),
                             _flat(ubx, P.n, "ubx"), _flat(lbg, P.mg, "lbg"), _flat(ubg, P.mg, "ubg"))
        st = int(o["status"][0])
        self._stats = dict(return_status=_cabi.STATUS.get(st, str(st)), success=st in (0, 1),
                           iter_count=int(o["iters"][0]), kkt_error=float(o["stats"][0, 0]))
        lam_p = np.zeros(P.np_)
        if P.np_:
            # dL/dp with L = f + lam_g'g: the initial-condition rows are X_0 - p[0:ns]; the cost holds xs = p[ns:] in
            # sum_{k<N} (X_k - xs)'Q(X_k - xs)  (centralized_six_robots_implementation.py:278,314)
            lam_p[:P.ns] = -o["lam_g"][0, :P.ns]
            Xk = o["x"][0, :P.ns * (P.N + 1)].reshape(P.N + 1, P.ns)[:P.N]
            Qd = np.tile(np.asarray(list(P.desc.Q), float), P.Nr)
            pv = np.asarray(_flat(p, P.np_, "p"))
            if getattr(P, "tracking", False):
                # Z[k] = [xr_k; ur_k] enters only the cost (X_k - xr_k)'Q(X_k - xr_k) + (U_k - ur_k)'R(U_k - ur_k)
                Z = pv[P.ns:P.ns + P.N * (P.ns + P.nc)].reshape(P.N, P.ns + P.nc)
                Uk = o["x"][0, P.ns * (P.N + 1):].reshape(P.N, P.nc)
                Rd = np.tile(np.asarray(list(P.desc.R), float), P.Nr)
                lam_z = np.concatenate([-2.0 * Qd * (Xk - Z[:, :P.ns]), -2.0 * Rd * (Uk - Z[:, P.ns:])], axis=1)
                lam_p[P.ns:P.ns + lam_z.size] = lam_z.ravel()
            else:
                lam_p[P.ns:2 * P.ns] = -2.0 * Qd * (Xk - pv[P.ns:2 * P.ns][None]).sum(axis=0)
            if getattr(P, "moving", False):
                # obstacle block O[k][o] = (ox, oy, c): row (k, i, o) = rho - c with rho = |pos_{k,i} - (ox, oy)|, so
                # dL/d(ox, oy) = -sum_i lam (pos - o) / rho and dL/dc = -sum_i lam
                o0 = P.np_ - 3 * P.N * P.nobs      # after xs (6Nr), or after Z with tracking_obstacles (3Nr + 5Nr N)
                O = pv[o0:].reshape(P.N, P.nobs, 3)
                lam = o["lam_g"][0, P.ns:].reshape(P.N, P.ns + P.M + P.Nr * P.nobs)[:, P.ns + P.M:].reshape(P.N, P.Nr, P.nobs)
                d = Xk.reshape(P.N, P.Nr, 3)[:, :, None, :2] - O[:, None, :, :2]
                gxy = d / np.linalg.norm(d, axis=-1, keepdims=True)
                lam_o = np.empty((P.N, P.nobs, 3))
                lam_o[..., :2] = -(lam[..., None] * gxy).sum(axis=1)
                lam_o[..., 2] = -lam.sum(axis=1)
                lam_p[o0:] = lam_o.ravel()
        return {"x": DM(o["x"][0]), "f": DM(o["f"][:1]), "g": DM(o["g"][0]), "lam_x": DM(o["lam_x"][0]),
                "lam_g": DM(o["lam_g"][0]), "lam_p": DM(lam_p)}

    def stats(self):
        return dict(self._stats)


_IPOPT_KEYS = {f[0] for f in _cabi.Opts._fields_}


def nlpsol(name, plugin, nlp, opts=None):
    """Drop-in for casadi.nlpsol(name, 'ipopt', nlp_prob, opts) (:345-346).

    `nlp` is a problem descriptor instead of CasADi's symbolic dict:
        {'family': 'unicycle_centralized', 'Nr', 'N', 'T', 'Q': (3,), 'R': (2,)}
        {'family': 'unicycle_obstacles', ..., 'obstacles': [[x, y, clearance], ...]}
        {'family': 'unicycle_moving_obstacles', ..., 'n_obs'}: the obstacles in p = [x0bar; xs; O[N][n_obs][3]]
        {'family': 'unicycle_tracking', 'Nr', 'N', 'T', 'Q', 'R'}: a per-stage reference in p = [x0bar; Z[N][5Nr]]
        {'family': 'unicycle_tracking_obstacles', ..., 'n_obs'}: both, p = [x0bar; Z[N][5Nr]; O[N][n_obs][3]]
    `opts` uses the reference's layout: {'print_time': 0, 'ipopt': {'max_iter': 2000, ...}}.
    """
    if plugin not in ("ipopt", "b200ipm"):
        raise ValueError("plugin %r: this library implements the interior-point path only" % (plugin,))
    if isinstance(nlp, dict) and nlp.get("family") == "van_der_pol":
        ip = dict((opts or {}).get("ipopt", {}))
        kw = {k: v for k, v in ip.items() if k in _IPOPT_KEYS}
        return NlpSolver(name, SmallOcp("van_der_pol", nlp.get("N", 20), nlp.get("T", 10.0), nlp.get("rk_steps", 4), **kw))
    if not isinstance(nlp, dict) or nlp.get("family", "unicycle_centralized") not in ("unicycle_centralized", "unicycle_obstacles",
                                                                                   "unicycle_moving_obstacles", "unicycle_tracking",
                                                                                   "unicycle_tracking_obstacles"):
        raise ValueError("nlp must be a descriptor {'family':'unicycle_centralized'|'unicycle_obstacles'|"
                         "'unicycle_moving_obstacles'|'unicycle_tracking'|'unicycle_tracking_obstacles','Nr','N','T',...}")
    for fam in ("unicycle_moving_obstacles", "unicycle_tracking_obstacles"):
        if nlp.get("family") == fam and nlp.get("n_obs") is None:
            raise ValueError("family '%s' needs 'n_obs'" % fam)
    if nlp.get("family") == "unicycle_obstacles" and nlp.get("obstacles") is None:
        raise ValueError("family 'unicycle_obstacles' needs 'obstacles': [[x, y, clearance], ...]")
    ip = dict((opts or {}).get("ipopt", {}))
    ip.update({k: v for k, v in (opts or {}).items() if k in _IPOPT_KEYS})
    kw = {k: v for k, v in ip.items() if k in _IPOPT_KEYS}          # print_level etc. are accepted and ignored
    prob = Problem(nlp["Nr"], nlp["N"], nlp["T"], nlp.get("Q", (1.0, 5.0, 0.1)), nlp.get("R", (0.5, 0.05)),
                   obstacles=nlp.get("obstacles") if nlp.get("family") == "unicycle_obstacles" else None,
                   moving_obstacles=nlp.get("n_obs") if nlp.get("family") == "unicycle_moving_obstacles" else None,
                   tracking=nlp.get("family") == "unicycle_tracking",
                   tracking_obstacles=nlp.get("n_obs") if nlp.get("family") == "unicycle_tracking_obstacles" else None, **kw)
    return NlpSolver(name, prob)
