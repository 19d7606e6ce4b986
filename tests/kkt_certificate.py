"""Solver-independent KKT certificate of a returned (x, lam_x, lam_g) -- TEST INFRASTRUCTURE ONLY.

Checks, in float64 on the NumPy restatements of the NLPs (UnicycleNLP, TrackingNLP, ObstacleNLP, StageObstacleNLP, VdpNLP),
that a point and its multipliers form a first-order KKT point in CasADi's conventions:

    grad f(x) + J(x)' lam_g + lam_x = 0
    lam_x <= 0 at an active lower bound, >= 0 at an active upper bound, == 0 (exactly) where a variable has no finite bound
    lam_g <= 0 on rows with only a lower bound, >= 0 on rows with only an upper bound, ~ 0 on the centralized block-0 rows
    |lam| * (distance to the bound it pushes against) ~ 0

It uses nothing of the solver that produced the point: not its dual residual, not its stopping test.  The tolerances
follow the solver's own stopping test restated in unscaled quantities: IPOPT scales the objective by
df = min(1, nlp_scaling_max_gradient / max|grad f(x0)|) and divides the dual infeasibility by
s_d = max(s_max, (sum|y| + sum|z|) / (m + n_bounds)) / s_max (ipm_driver.cuh), so a point it accepts at tol has an unscaled
stationarity residual <= tol s_d / df.  s_d is recomputed here from the returned multipliers times df.
"""
import numpy as np

from oracle.nlp_numpy import UnicycleNLP
from oracle.vdp_nlp import VdpNLP

S_MAX = 100.0


def objective_scaling(nlp, x0, p=None, lbx=None, ubx=None, max_gradient=100.0):
    """df = min(1, max_gradient / max|grad f(x0)|), floored at 1e-8 like the kernels; fixed variables (lbx == ubx) are
    parameters and do not count."""
    grad = derivatives(nlp, x0, p)[0]
    if lbx is not None:
        grad = grad[~(np.asarray(lbx) == np.asarray(ubx))]
    gmax = np.abs(grad).max() if grad.size else 0.0
    return max(max_gradient / gmax, 1e-8) if gmax > max_gradient else 1.0


def derivatives(nlp, x, p):
    """(grad f, g, dense J) at x.  VdpNLP has no derivatives of its own: central differences of fg."""
    x = np.asarray(x, float)
    if isinstance(nlp, VdpNLP):
        f0, g0 = nlp.fg(x)
        grad, J = np.empty(nlp.n), np.empty((nlp.mg, nlp.n))
        for j in range(nlp.n):
            h = 1e-6 * max(1.0, abs(x[j]))
            e = np.zeros(nlp.n); e[j] = h
            fp, gp = nlp.fg(x + e)
            fm, gm = nlp.fg(x - e)
            grad[j] = (fp - fm) / (2 * h)
            J[:, j] = (gp - gm) / (2 * h)
        return grad, g0, J
    return nlp.grad_f(x, p), nlp.g(x, p), nlp.jac_g(x, p)


def dummy_rows(nlp):
    """Rows with a constant value and no Jacobian: the pair rows of block 0 of the centralized family (g = 3.5)."""
    mask = np.zeros(nlp.mg, bool)
    if isinstance(nlp, UnicycleNLP):
        mask[nlp.ns:nlp.blk] = True
    return mask


def _one_sided(v, lam, lo, hi, relax):
    """Per entry: the multiplier's part pushing against each bound, the distance to it and the activity of the bound."""
    eq = lo == hi          # equality rows and fixed variables: no complementarity, no sign condition
    fl, fu = np.isfinite(lo) & ~eq, np.isfinite(hi) & ~eq
    lo_f, hi_f = np.where(fl, lo, 0.0), np.where(fu, hi, 0.0)
    # distances to the bounds relaxed by relax * max(1, |b|), the bounds IPOPT works with (bound_relax_factor)
    gap_l = np.where(fl, v - (lo_f - relax * np.maximum(1.0, np.abs(lo_f))), np.inf)
    gap_u = np.where(fu, hi_f + relax * np.maximum(1.0, np.abs(hi_f)) - v, np.inf)
    act_l, act_u = 1e-6 * np.maximum(1.0, np.abs(lo_f)), 1e-6 * np.maximum(1.0, np.abs(hi_f))
    active_l = fl & (gap_l <= act_l) & ~(fu & (gap_u <= act_u))
    active_u = fu & (gap_u <= act_u) & ~(fl & (gap_l <= act_l))
    lam_l, lam_u = np.maximum(-lam, 0.0), np.maximum(lam, 0.0)
    compl = np.concatenate([lam_l * np.abs(np.where(fl, gap_l, 0.0)), lam_u * np.abs(np.where(fu, gap_u, 0.0))])
    tol_eq = relax * np.maximum(1.0, np.abs(np.where(eq, lo, 0.0)))
    viol = np.maximum(np.maximum(np.where(fl, -gap_l, -np.inf), np.where(fu, -gap_u, -np.inf)),
                      np.where(eq, np.abs(v - np.where(eq, lo, 0.0)) - tol_eq, -np.inf))
    # the multiplier may only push against a bound that exists; at an active bound only against that bound
    wrong = np.concatenate([np.where(~fl & ~eq, lam_l, 0.0), np.where(~fu & ~eq, lam_u, 0.0),
                            np.where(active_l, lam_u, 0.0), np.where(active_u, lam_l, 0.0)])
    return compl, viol, wrong


def measure(nlp, x, lam_x, lam_g, p, lbx, ubx, lbg, ubg, df, relax=1e-8, feas=None):
    """The certificate's quantities (unscaled unless named *_scaled).  feas: the tolerance of the constraint rows' feasibility
    (default relax); a solver stops with |g - s| <= tol, so with bound_relax_factor < tol a row may miss its bound by tol."""
    x, lam_x, lam_g = (np.asarray(a, float).reshape(-1) for a in (x, lam_x, lam_g))
    lbx, ubx, lbg, ubg = (np.asarray(a, float).reshape(-1) for a in (lbx, ubx, lbg, ubg))
    grad, g, J = derivatives(nlp, x, p)
    dummy = dummy_rows(nlp)
    stat = grad + J.T @ lam_g + lam_x
    free = ~np.isfinite(lbx) & ~np.isfinite(ubx)
    rows = ~dummy & (np.isfinite(lbg) | np.isfinite(ubg))
    ineq = rows & (lbg != ubg)
    cx, vx, wx = _one_sided(x, lam_x, lbx, ubx, relax)
    cg, vg, wg = _one_sided(g[~dummy], lam_g[~dummy], lbg[~dummy], ubg[~dummy], relax)
    if feas is not None:
        vg = _one_sided(g[~dummy], lam_g[~dummy], lbg[~dummy], ubg[~dummy], feas)[1]
    # IPOPT's scaling of the dual infeasibility and of the complementarity (ipm_driver.cuh), from the scaled multipliers
    nzb = np.isfinite(lbx).sum() + np.isfinite(ubx).sum() + np.isfinite(lbg[ineq]).sum() + np.isfinite(ubg[ineq]).sum()
    ysum = df * np.abs(lam_g[rows]).sum()
    zsum = df * (np.abs(lam_x[~free]).sum() + np.abs(lam_g[ineq]).sum())
    s_d = max(S_MAX, (ysum + zsum) / max(1.0, rows.sum() + nzb)) / S_MAX
    s_c = max(S_MAX, zsum / max(1.0, nzb)) / S_MAX
    stat_inf = np.abs(stat).max()
    compl = max(cx.max(initial=0.0), cg.max(initial=0.0))
    pinf = max(0.0, vx.max(initial=0.0), vg.max(initial=0.0))
    return dict(stat=stat_inf, grad=np.abs(grad).max(), lam_max=max(np.abs(lam_x).max(), np.abs(lam_g).max()), s_d=s_d, s_c=s_c, df=df, pinf=pinf, compl=compl,
                wrong_sign=max(wx.max(initial=0.0), wg.max(initial=0.0)),
                free_lam=np.abs(lam_x[free]).max(initial=0.0), dummy_lam=np.abs(lam_g[dummy]).max(initial=0.0),
                scaled_err=max(df * stat_inf / s_d, pinf, df * compl / s_c))


def certify(nlp, x, lam_x, lam_g, p, lbx, ubx, lbg, ubg, df, relax=1e-8, tol=1e-8, feas=None):
    """Assert that (x, lam_x, lam_g) is a KKT point of the NLP at tolerance tol; return the measured quantities."""
    m = measure(nlp, x, lam_x, lam_g, p, lbx, ubx, lbg, ubg, df, relax, feas)
    stat_tol = 2 * tol * m["s_d"] / df + 1e-11 * (1.0 + m["grad"])
    sign_tol = 10 * tol / df
    compl_tol = max(1e-7, 2 * tol * m["s_c"] / df)
    assert m["stat"] <= stat_tol, ("stationarity", m["stat"], stat_tol, m)
    assert m["pinf"] <= 0.0, ("primal feasibility", m["pinf"], m)
    assert m["free_lam"] == 0.0, ("lam_x of a variable without finite bounds", m["free_lam"])
    assert m["wrong_sign"] <= sign_tol, ("multiplier sign", m["wrong_sign"], sign_tol, m)
    assert m["dummy_lam"] <= sign_tol, ("lam_g of the block-0 rows", m["dummy_lam"], sign_tol)
    assert m["compl"] <= compl_tol, ("complementarity", m["compl"], compl_tol, m)
    return m
