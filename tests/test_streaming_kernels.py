"""The streaming kernels either side of the solver at the batch sizes they run at: K1 nmpc_eval (every one of its 20 kernels),
nmpc_shift, nmpc_plant and nmpc_advanced_step, with more points than CTAs, against the high-precision references of
tests/streaming_ref.py.

At B = 37 every CTA of eval_kernel evaluates one point; at the sizes the bandwidth figures are quoted for, each CTA walks
through many, with a register prefetch of the next point, an asynchronous bulk write-back of the record and a shifted shared
image of g whenever the global row is not 16-byte aligned.  Here every kernel runs with several points per CTA and an uneven
last round, and is held to:
  * the reference, entry by entry, to k eps S (S: the sum of the absolute values of the terms of the entry's expression);
  * the same bits for a point evaluated alone, in a batch smaller than the grid, in reversed order and as the k-th point of
    its CTA (the arithmetic of one point does not depend on where or when it runs);
  * the same bits with outputs or inputs at an 8-byte offset and with any subset of the outputs requested;
  * guard elements before and after every output that stay untouched, and no element of [0, B) left unwritten;
  * NaN / Inf in one point that stays in that point, also for the clean point that follows it in the same CTA.
"""
import ctypes as C

import numpy as np
import pytest

from oracle.nlp_numpy import UnicycleNLP, euler_plant, shift_warm_start
from oracle.oracle_lib import Oracle
from tests import advanced_step_ref as AR
from tests import streaming_ref as SR
from tests.tracking_ref import TrackingNLP, TrackingOracle

T = 0.3
Q, R = (1.0, 5.0, 0.1), (0.5, 0.05)
EDGE_TH = [0.0, -0.0, np.pi / 2, -np.pi / 2, np.pi, 1e3, 1e6, -1e15]     # -1e15: Payne-Hanek reduction in sin / cos
FILL = 0x7FF8DEADBEEF0001          # NaN with a payload: the fill of every output buffer, compared as int64 bits
NMPC_EINVAL = -1

# One shape per eval_kernel instantiation and layout (the cheapest at 148 SMs), plus the benchmark shape (6, 20) whose g row
# (mg = 693) is odd, so that its shared image alternates between its two positions from point to point.
# (tracking, Nr, N): variant and grid at 148 SMs
SHAPES = {
    (False, 1, 1): (1, 44252), (False, 5, 19): (2, 740), (False, 6, 22): (3, 444), (False, 6, 20): (3, 592),
    (False, 7, 23): (4, 296), (False, 2, 126): (5, 296), (False, 5, 57): (6, 148), (False, 3, 114): (7, 148),
    (False, 2, 190): (8, 148), (False, 12, 20): (0, 148), (False, 16, 20): ("big", 1184),
    (True, 1, 1): (1, 43364), (True, 6, 13): (2, 740), (True, 8, 13): (3, 444), (True, 4, 47): (4, 296),
    (True, 2, 111): (5, 296), (True, 7, 32): (6, 148), (True, 2, 167): (7, 148), (True, 29, 3): (8, 148),
    (True, 12, 20): (0, 148), (True, 14, 22): ("big", 1184),
}


def _sid(s):
    return "%s-%dx%d" % ("trk" if s[0] else "set", s[1], s[2])


def _batch(variant, grid):
    """3 grid + r (2 grid + r for eval_kernel_big), 0 < r < grid: several points per CTA and an uneven last round."""
    return (2 if variant == "big" else 3) * grid + max(7, grid // 3 + 1)


def _points(rng, d, B, edges):
    """Random points, and at the indices `edges` the edge block: theta over EDGE_TH, v = om = 0, lam = 0, |w| up to 1e6."""
    n, mg, nX = d["n"], d["mg"], d["nX"]
    W = rng.normal(scale=2.0, size=(B, n))
    W[:, 2:nX:3] = rng.uniform(-10.0, 10.0, size=(B, nX // 3))
    P, LAM = rng.normal(size=(B, d["np"])), rng.normal(size=(B, mg))
    for e, b in enumerate(edges):
        if e % 4 == 1:
            W[b, nX:] = 0.0
        elif e % 4 == 2:
            LAM[b] = 0.0
        elif e % 4 == 3:
            W[b], P[b], LAM[b] = (rng.uniform(-1e6, 1e6, size=a.shape[1]) for a in (W, P, LAM))
        W[b, 2:nX:3] = np.resize(np.roll(EDGE_TH, e), nX // 3)
    return W, P, LAM


def _ref_of(orc_like, Nr, N, tracking):
    return SR.EvalRef(Nr, N, T, Q, R, tracking, orc_like.jac_pattern(), orc_like.hess_pattern())


# ------------------------------------------------------------------------------------------------------------------------
# CPU: the reference, its rounding error, the checker and the shape table
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tracking", [False, True], ids=["setpoint", "tracking"])
@pytest.mark.parametrize("Nr,N", [(1, 3), (2, 2), (3, 4), (4, 2)])
def test_reference_matches_oracle_and_numpy(tracking, Nr, N):
    """EvalRef against orc_eval (the C oracle; its tracking derivation for the tracking layout) and against the dense
    UnicycleNLP / TrackingNLP jac_g and hess_lag read at the pattern's slots, to 1e-13."""
    orc = (TrackingOracle if tracking else Oracle)(Nr, N, T, Q=Q, R=R)
    nlp = (TrackingNLP if tracking else UnicycleNLP)(Nr, N, T, Q, R)
    d = SR.dims(Nr, N, tracking)
    assert (d["n"], d["mg"], d["nnzj"], d["nnzh"]) == (orc.n, orc.mg, orc.nnz_jac, orc.nnz_hess)
    rng = np.random.default_rng(100 * Nr + N + tracking)
    B = 12
    W, P, LAM = _points(rng, d, B, edges=range(0, B, 2))
    ref = _ref_of(orc, Nr, N, tracking).eval(W, P, LAM)
    jcp, jri = orc.jac_pattern()
    hcp, hri = orc.hess_pattern()
    jcol, hcol = np.repeat(np.arange(d["n"]), np.diff(jcp)), np.repeat(np.arange(d["n"]), np.diff(hcp))
    close = lambda a, b, what: np.testing.assert_allclose(a, b, rtol=1e-13, atol=1e-13, err_msg=what)
    for b in range(B):
        e = orc.eval(W[b], P[b], LAM[b])
        close(ref["f"][0][b], e["f"], "f vs orc_eval")
        for k in ("grad", "g", "jac", "hess"):
            close(ref[k][0][b], e[k], k + " vs orc_eval")
        close(ref["f"][0][b], nlp.f(W[b], P[b]), "f vs NumPy")
        close(ref["grad"][0][b], nlp.grad_f(W[b], P[b]), "grad vs NumPy")
        close(ref["g"][0][b], nlp.g(W[b], P[b]), "g vs NumPy")
        close(ref["jac"][0][b], nlp.jac_g(W[b], P[b])[jri, jcol], "jac vs NumPy")
        close(ref["hess"][0][b], nlp.hess_lag(W[b], P[b], LAM[b])[hri, hcol], "hess vs NumPy")


def _mp(a):
    import mpmath
    return np.frompyfunc(mpmath.mpf, 1, 1)(np.asarray(a, np.float64))


def _mp_excess(val, exact, S, k):
    """excess() with the difference taken in 50 digits (no rounding of the exact value to double first)."""
    diff = np.abs(_mp(val) - exact)
    return SR.excess(diff.astype(np.float64), np.zeros(np.shape(val)), S, k)


@pytest.mark.parametrize("tracking", [False, True], ids=["setpoint", "tracking"])
def test_reference_rounding_against_mpmath(tracking):
    """The float64 reference is within 2 eps S of the same expressions evaluated in 50 digits, at theta = 0, -0.0, +-pi/2,
    pi, 1e3, 1e6, -1e15 and v = 0: the bound the GPU tests use has its own error inside it."""
    import mpmath
    mpmath.mp.dps = 50
    Nr, N = 3, 2
    d = SR.dims(Nr, N, tracking)
    orc = Oracle(Nr, N, T, Q=Q, R=R)          # the tracking handle has the setpoint handle's patterns
    ref = _ref_of(orc, Nr, N, tracking)
    rng = np.random.default_rng(7)
    W, P, LAM = _points(rng, d, 8, edges=range(8))
    W[0, d["nX"]:] = 0.0
    fl = ref.eval(W, P, LAM)
    ex = ref.eval(_mp(W), _mp(P), _mp(LAM), sin=np.frompyfunc(mpmath.sin, 1, 1), cos=np.frompyfunc(mpmath.cos, 1, 1))
    worst = {}
    for k in ("grad", "g", "jac", "hess"):
        worst[k] = _mp_excess(fl[k][0], ex[k][0], fl[k][1], 2.0)
    worst["f"] = _mp_excess(fl["f"][0], ex["f"][0], fl["f"][1], 2.0)
    print("reference / 50 digits, error over 2 eps S:", worst)
    assert max(worst.values()) <= 1.0, worst
    # the plant's reference likewise
    st = rng.normal(size=(8, 3 * Nr))
    st[:, 2::3] = np.resize(EDGE_TH, (8, Nr))
    a, S = SR.plant(st, W, Nr, N, T)
    e, _ = SR.plant(_mp(st), _mp(W), Nr, N, T, sin=np.frompyfunc(mpmath.sin, 1, 1), cos=np.frompyfunc(mpmath.cos, 1, 1))
    assert _mp_excess(a, e, S, 2.0) <= 1.0


def test_checker_rejects_corruptions():
    """The comparison the GPU tests make accepts the oracle's record and rejects each of: one Jacobian value written to its
    neighbouring slot, two Hessian slots swapped, the last element of g left at the fill, point b's record replaced by point
    b+1's, and f missing one work item's share of the cost."""
    Nr, N, B = 3, 4, 6
    orc = Oracle(Nr, N, T, Q=Q, R=R)
    d = SR.dims(Nr, N, False)
    W, P, LAM = _points(np.random.default_rng(11), d, B, edges=[0])
    rec = {k: np.zeros((B,) + s) for k, s in (("f", ()), ("grad", (d["n"],)), ("g", (d["mg"],)), ("jac", (d["nnzj"],)),
                                              ("hess", (d["nnzh"],)))}
    for b in range(B):
        e = orc.eval(W[b], P[b], LAM[b])
        for k in rec:
            rec[k][b] = e[k]
    er = _ref_of(orc, Nr, N, False)
    ref = er.eval(W, P, LAM)
    ok = SR.record_excess(ref, rec)
    assert max(ok.values()) <= 1.0, ok
    b = 2
    tvs = er.jac_kinds["Tvs"][0][0]                      # a T v sin(theta) slot; its neighbour holds -T cos(theta)
    hs_tt, hs_vt = er.hess_kinds["tt"][0][0], er.hess_kinds["vt"][0][0]
    ix, iu = (N - 1) * d["ns"] + 3 * (Nr - 1), d["nX"] + (N - 1) * d["nc"] + 2 * (Nr - 1)     # item (k, i) = (N - 1, Nr - 1)
    dropped = sum(Q[c] * (W[b, ix + c] - P[b, d["ns"] + 3 * (Nr - 1) + c]) ** 2 for c in range(3)) + \
        sum(R[c] * W[b, iu + c] ** 2 for c in range(2))

    def moved(r):
        r["jac"][b, tvs + 1] = r["jac"][b, tvs]

    def swapped(r):
        r["hess"][b, [hs_tt, hs_vt]] = r["hess"][b, [hs_vt, hs_tt]]

    def fill(r):
        r["g"][b, -1] = np.int64(FILL).view(np.float64)

    def neighbour(r):
        for k in r:
            r[k][b] = r[k][b + 1]

    def f_short(r):
        r["f"][b] -= dropped

    for corrupt in (moved, swapped, fill, neighbour, f_short):
        bad = {k: v.copy() for k, v in rec.items()}
        corrupt(bad)
        ex = SR.record_excess(ref, bad)
        assert max(ex.values()) > 1.0, (corrupt.__name__, ex)


def test_shape_table_covers_every_instantiation():
    """The mirror of nmpc_eval's launch selection puts SHAPES on all 20 kernels (PF 0..8 of eval_kernel and eval_kernel_big,
    setpoint and tracking), with the grids stated at 148 SMs; the shapes have odd and even n, mg and nnz_jac, which select
    the different write-back branches; the sizes the mirror uses are the oracle's."""
    seen = set()
    for (tracking, Nr, N), (variant, grid) in SHAPES.items():
        v, g, smem = SR.eval_launch(Nr, N, tracking, 148)
        assert (v, g) == (variant, grid), ((tracking, Nr, N), v, g)
        assert (v == "big") == (smem > 220 * 1024)
        B = _batch(v, g)
        assert 0 < B - (2 if v == "big" else 3) * g < g
        seen.add((tracking, v))
        if not tracking:
            orc = Oracle(Nr, N, T)
            d = SR.dims(Nr, N, False)
            assert (d["n"], d["mg"], d["nnzj"], d["nnzh"]) == (orc.n, orc.mg, orc.nnz_jac, orc.nnz_hess)
    assert seen == {(t, v) for t in (False, True) for v in list(range(9)) + ["big"]}
    for key in ("n", "mg", "nnzj"):
        assert {SR.dims(Nr, N, t)[key] % 2 for t, Nr, N in SHAPES} == {0, 1}, key
    # the benchmark shape: odd mg, so its g rows alternate between 16-byte-aligned and 8-byte-offset starts
    assert SR.dims(6, 20, False)["mg"] == 693


@pytest.mark.parametrize("Nr,N", [(1, 1), (3, 1), (2, 2), (3, 20), (6, 20)])
def test_shift_and_plant_references_match_oracle(Nr, N):
    orc, nlp = Oracle(Nr, N, T), UnicycleNLP(Nr, N, T)
    rng = np.random.default_rng(Nr * 7 + N)
    W = rng.normal(size=(5, orc.n))
    st = rng.normal(size=(5, 3 * Nr))
    st[:, 2::3] = np.resize(EDGE_TH, (5, Nr))
    sh = SR.shift(W, Nr, N)
    pl, _ = SR.plant(st, W, Nr, N, T)
    nX = 3 * Nr * (N + 1)
    for b in range(5):
        np.testing.assert_array_equal(sh[b], shift_warm_start(nlp, W[b]))
        np.testing.assert_array_equal(sh[b], orc.shift(W[b]))
        np.testing.assert_array_equal(pl[b], euler_plant(nlp, st[b], W[b, nX:nX + 2 * Nr]))
        np.testing.assert_allclose(pl[b], orc.plant(st[b], W[b, nX:nX + 2 * Nr]), rtol=1e-15, atol=0)


# ------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _t(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")


class _Out:
    """A [B, m] output inside a buffer filled with FILL: `off` guard elements before it (2: the output is 16-byte aligned,
    1: at an 8-byte offset) and one guard row after it."""

    def __init__(self, torch, B, m, off):
        self.torch, self.B, self.m, self.off = torch, B, m, off
        self.buf = torch.empty(off + (B + 1) * m, dtype=torch.float64, device="cuda")
        assert self.buf.data_ptr() % 16 == 0
        self.buf.view(torch.int64).fill_(FILL)
        self.t = self.buf[off:off + B * m].view(B, m)

    def check(self, what):
        bits = self.buf.view(self.torch.int64)
        end = self.off + self.B * self.m
        assert bool((bits[:self.off] == FILL).all()) and bool((bits[end:] == FILL).all()), "%s: written outside [0, B)" % what
        assert not bool((bits[self.off:end] == FILL).any()), "%s: an element of [0, B) was never written" % what


def _at_offset(torch, t):
    """A copy of t whose data starts 8 bytes past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 1, dtype=torch.float64, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 8
    return v


def _bits(torch, t):
    return t.contiguous().view(torch.int64)


def _same(torch, a, b):
    return torch.equal(_bits(torch, a), _bits(torch, b))


WIDTH = lambda prob: dict(f=1, grad=prob.n, g=prob.mg, jac=prob.nnz_jac, hess=prob.nnz_hess)
ALL = ("f", "grad", "g", "jac", "hess")


def _eval(torch, prob, w, p, lam, want=ALL, off=2):
    """nmpc_eval through the C ABI into guarded outputs; returns (rc, {name: _Out})."""
    B, wd = w.shape[0], WIDTH(prob)
    outs = {k: _Out(torch, B, wd[k], off) for k in want}
    ptr = lambda k: outs[k].t.data_ptr() if k in outs else None
    rc = prob.L.nmpc_eval(prob.h, B, w.data_ptr(), p.data_ptr(), None if lam is None else lam.data_ptr(), ptr("f"), ptr("grad"),
                          ptr("g"), ptr("jac"), ptr("hess"), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, outs


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPES), ids=_sid)
def test_eval_kernel_streaming(pkg, torch_cuda, shape):
    torch = torch_cuda
    tracking, Nr, N = shape
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    variant, grid, _ = SR.eval_launch(Nr, N, tracking, sm)
    B = _batch(variant, grid)
    assert SR.eval_launch(Nr, N, tracking, sm, B)[1] == grid < B
    prob = pkg.Problem(Nr, N, T, Q, R, tracking=tracking)
    d = SR.dims(Nr, N, tracking)
    assert (prob.n, prob.mg, prob.np_, prob.nnz_jac, prob.nnz_hess) == (d["n"], d["mg"], d["np"], d["nnzj"], d["nnzh"])
    rng = np.random.default_rng(sum(shape) * 31 + tracking)
    E = 16
    W, P, LAM = _points(rng, d, B, edges=list(range(E)) + list(range(B - E, B)))
    w, p, lam = _t(torch, W), _t(torch, P), _t(torch, LAM)

    rc, full = _eval(torch, prob, w, p, lam)
    assert rc == 0, prob.L.nmpc_last_error()
    for k, o in full.items():
        o.check(k)

    # against the reference, in chunks of points
    ref = SR.EvalRef(Nr, N, T, Q, R, tracking, prob.jac_pattern(), prob.hess_pattern())
    chunk = max(1, 4_000_000 // (2 * d["n"] + d["mg"] + d["nnzj"] + d["nnzh"]))
    worst = dict.fromkeys(ALL, 0.0)
    for c0 in range(0, B, chunk):
        c1 = min(B, c0 + chunk)
        dev = {k: o.t[c0:c1].cpu().numpy() for k, o in full.items()}
        dev["f"] = dev["f"][:, 0]
        ex = SR.record_excess(ref.eval(W[c0:c1], P[c0:c1], LAM[c0:c1]), dev)
        worst = {k: max(worst[k], ex[k]) for k in worst}
    print("\neval %s variant %s: sm %d grid %d B %d  error / bound %s" % (_sid(shape), variant, sm, grid, B,
                                                                          {k: round(v, 3) for k, v in worst.items()}))
    assert max(worst.values()) <= 1.0, worst

    def same_rows(outs, rows):
        for k, o in outs.items():
            assert _same(torch, o.t, full[k].t[rows]), k

    # bitwise invariance: alone, one point per CTA, reversed order (every point moves to another CTA and position)
    for b in sorted({0, 1, grid - 1, grid, 2 * grid + 1, B - 1}):
        rc, one = _eval(torch, prob, w[b:b + 1], p[b:b + 1], lam[b:b + 1])
        assert rc == 0
        same_rows(one, slice(b, b + 1))
    m = min(grid - 1, 97)
    rc, few = _eval(torch, prob, w[grid:grid + m], p[grid:grid + m], lam[grid:grid + m])
    assert rc == 0
    same_rows(few, slice(grid, grid + m))
    rc, rev = _eval(torch, prob, w.flip(0).contiguous(), p.flip(0).contiguous(), lam.flip(0).contiguous())
    assert rc == 0
    for k, o in rev.items():
        o.check(k + " reversed")
        assert _same(torch, o.t.flip(0), full[k].t), k

    # outputs at an 8-byte offset; inputs at an 8-byte offset
    rc, odd = _eval(torch, prob, w, p, lam, off=1)
    assert rc == 0
    for k, o in odd.items():
        o.check(k + " at offset")
    same_rows(odd, slice(0, B))
    rc, oin = _eval(torch, prob, _at_offset(torch, w), _at_offset(torch, p), _at_offset(torch, lam))
    assert rc == 0
    same_rows(oin, slice(0, B))

    # subsets of the outputs: each alone, g + jac without lam, grad + hess, lam with hess NULL (the two pairs at an 8-byte
    # offset); hess without lam is refused
    for want, with_lam in [((k,), k == "hess") for k in ALL] + [(("g", "jac"), False), (("grad", "hess"), True),
                                                                 (("f", "grad", "g", "jac"), True)]:
        rc, sub = _eval(torch, prob, w, p, lam if with_lam else None, want=want, off=1 if len(want) == 2 else 2)
        assert rc == 0, want
        for k, o in sub.items():
            o.check("%s of %s" % (k, want))
        same_rows(sub, slice(0, B))
    rc, _ = _eval(torch, prob, w, p, None, want=("hess",))
    assert rc == NMPC_EINVAL

    # NaN isolation: poisoned points first in their CTA (b < grid) and second (grid <= b < 2 grid), each followed by a clean
    # point of the same CTA (b + grid)
    bad = [1, 2, 3, grid + 4, grid + 5, grid + 6]
    wq, pq, lq = w.clone(), p.clone(), lam.clone()
    for j, b in enumerate(bad):
        if j % 3 == 0:
            wq[b, d["n"] // 2] = float("nan")
        elif j % 3 == 1:
            lq[b, d["mg"] // 2] = float("inf")
        else:
            pq[b, 0] = float("nan")
    rc, pois = _eval(torch, prob, wq, pq, lq)
    assert rc == 0
    clean = torch.ones(B, dtype=torch.bool, device="cuda")
    clean[bad] = False
    for k, o in pois.items():
        o.check(k + " poisoned")
        assert _same(torch, o.t[clean], full[k].t[clean]), k


@pytest.mark.gpu
@pytest.mark.parametrize("Nr", [3, 6])
@pytest.mark.parametrize("N", [1, 2, 20])
def test_shift_kernel_streaming(pkg, torch_cuda, Nr, N):
    """nmpc_shift bit for bit against the NumPy shift, one instance and 3 x 8 sm_count + 7 (beyond its grid of 8 sm_count
    CTAs); aligned (the 128-bit path at even Nr) and with the input or the output at an 8-byte offset (the scalar path)."""
    torch = torch_cuda
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    prob = pkg.Problem(Nr, N, T)
    rng = np.random.default_rng(Nr * 100 + N)
    for B in (1, 3 * 8 * sm + 7):
        W = rng.normal(size=(B, prob.n))
        ref = SR.shift(W, Nr, N)
        w = _t(torch, W)
        for in_off, out_off in ((False, 2), (True, 2), (False, 1)):
            o = _Out(torch, B, prob.n, out_off)
            pkg._cabi.check(prob.L.nmpc_shift(prob.h, B, (_at_offset(torch, w) if in_off else w).data_ptr(), o.t.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream))
            torch.cuda.synchronize()
            o.check("shift B=%d in_off=%s out_off=%d" % (B, in_off, out_off))
            np.testing.assert_array_equal(o.t.cpu().numpy().view(np.int64), ref.view(np.int64))


@pytest.mark.gpu
def test_plant_kernel_streaming(pkg, torch_cuda):
    """nmpc_plant with B Nr above its grid of 16 sm_count x 256 threads, theta edge values included: within
    4 eps (|x| + |T v cos theta|) per component of the float64 reference."""
    torch = torch_cuda
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    Nr, N = 2, 1
    B = 16 * sm * 256 // Nr + 4099
    assert B * Nr > 16 * sm * 256
    prob = pkg.Problem(Nr, N, T)
    rng = np.random.default_rng(5)
    st = rng.normal(scale=3.0, size=(B, 3 * Nr))
    st[:, 2::3] = rng.uniform(-10.0, 10.0, size=(B, Nr))
    st[:64, 2::3] = np.resize(EDGE_TH, (64, Nr))
    st[-64:, 2::3] = np.resize(EDGE_TH[::-1], (64, Nr))
    xo = rng.normal(size=(B, prob.n))
    xo[::5, 3 * Nr * (N + 1):] = 0.0
    ref, S = SR.plant(st, xo, Nr, N, T)
    for off in (2, 1):
        o = _Out(torch, B, 3 * Nr, off)
        pkg._cabi.check(prob.L.nmpc_plant(prob.h, B, _t(torch, st).data_ptr(), _t(torch, xo).data_ptr(), o.t.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        o.check("plant off=%d" % off)
        r = SR.excess(o.t.cpu().numpy(), ref, S, 4.0)
        print("\nplant: sm %d B %d Nr %d (B Nr = %d)  error / 4 eps S = %.3f" % (sm, B, Nr, B * Nr, r))
        assert r <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("batched", [False, True], ids=["shared_bounds", "per_instance_bounds"])
def test_advanced_step_kernel_streaming(pkg, torch_cuda, batched):
    """nmpc_advanced_step for six robots at B = 1,500 (B n above its grid of 8 sm_count x 256 threads) on a random jac, with
    mixed sens_status and finite and infinite bounds, against tests/advanced_step_ref.advanced_step at the tolerance of
    tests/test_advanced_step.py (1e-15 sum|jac||dx0| + 2 ulps; X_0 exact)."""
    torch = torch_cuda
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    Nr, N, B = 6, 20, 1500
    prob = pkg.Problem(Nr, N, T)
    ns, n = prob.ns, prob.n
    assert B * n > 8 * sm * 256
    rng = np.random.default_rng(17 + batched)
    lbx, ubx, _, _ = prob.bounds(0.3, 0.22, 2.84)
    if batched:
        s = rng.uniform(0.5, 1.5, size=(B, 1))
        lbx, ubx = lbx[None] * s, ubx[None] * s
        lbx[B // 2:, :ns] = -np.inf          # infinite position bounds on half the instances
    x = rng.uniform(-1.0, 1.0, size=(B, n)) * np.where(np.isfinite(ubx), np.abs(np.nan_to_num(ubx, posinf=1.0)), 3.0)
    x[::7, -1] = 3.0                         # a few components already outside their bound: never pulled further out
    jac = rng.normal(size=(B, ns, n))
    P = rng.normal(size=(B, prob.np_))
    meas = P[:, :ns] + 0.05 * rng.normal(size=(B, ns))
    status = np.where(rng.uniform(size=B) < 0.2, rng.choice([1, -2], size=B), 0).astype(np.int32)
    ref = AR.advanced_step(x, jac, status, P, meas, lbx, ubx)
    o = _Out(torch, B, n, 2)
    tst = torch.as_tensor(status, device="cuda")
    args = [_t(torch, a) for a in (x, jac, P, meas, lbx, ubx)]
    pkg._cabi.check(prob.L.nmpc_advanced_step(prob.h, B, args[0].data_ptr(), args[1].data_ptr(), tst.data_ptr(), args[2].data_ptr(),
                                              args[3].data_ptr(), args[4].data_ptr(), args[5].data_ptr(), int(batched),
                                              o.t.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    o.check("advanced_step")
    xc = o.t.cpu().numpy()
    assert np.array_equal(xc[:, :ns], meas)
    keep = status != 0
    assert np.array_equal(xc[keep, ns:].view(np.int64), x[keep, ns:].view(np.int64))
    tol = 1e-15 * np.einsum("bjn,bj->bn", np.abs(jac), np.abs(meas - P[:, :ns])) + 2 * np.finfo(float).eps * np.abs(ref)
    assert np.all(np.abs(xc - ref) <= tol), np.abs(xc - ref).max()
    lo, hi = np.broadcast_to(lbx, (B, n)), np.broadcast_to(ubx, (B, n))
    assert ((xc == lo) | (xc == hi))[~keep].sum() > 0          # the clamp was exercised
