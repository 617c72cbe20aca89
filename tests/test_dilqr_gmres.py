"""GMRES for the adjoint system of the DiLQR backward (``solver="gmres"``).

The DiLQR backward solves A'w = g per problem.  The reference (fix_point_equ,
lqr_step_explicit.py:458-598) assembles A densely and calls linalg.solve; the package's default
solves it by Richardson iteration w <- g + M'w (M = I - A), which converges only where
rho(M) < 1.  ``solver="gmres"`` runs restarted GMRES per problem on the device instead.

``dilqr_backward_dense`` below is the reference's dense solve restated on the oracle's pieces:
A' is assembled column by column by applying the oracle's M' map (the KKT pass plus the
Dx / Du / d_x / d_u contraction of ``port.dilqr_backward``) to the unit vectors, batched along
the batch axis as fix_point_equ does, and solved by torch.linalg.solve in FP64.

CPU tests pin that dense oracle to the reference's goldens and show that the hard case
(``HARD``: cartpole, cold start, 10 iLQR iterations) is beyond Richardson: rho(M_b) > 1 for some
problem, and 30 Richardson passes still move w by more than 1e-2 (relative).

GPU tests (FP64 unless stated):
- at converged points GMRES equals Richardson run to 1e-14, on the fused, factored and generic
  paths, each case asserting the path it took; rocket (generic) equals the dense solve;
- on the hard case the device's w has a backward error |g - A'w| / |g| <= 1e-11 under the
  oracle's dense A', and dC, dc, dtheta agree with the dense solve per problem within
  10 cond(A_b) 1e-15 + 1e-10;
- g_b = 0 gives exact zeros, a short budget warns, a non-convex adjoint QP raises;
- a batch of 65541 problems tiled from 41 reproduces the base's w, gradients and per-problem
  iteration counts bit for bit;
- deferred and immediate modes, MPC and _solver, and the torch op agree bit for bit;
- FP32: backward error <= 1e-5 at a converged point, dtheta within 10x the FP32 oracle's own
  error."""
import importlib
import warnings
from collections import namedtuple

import pytest
import torch

from common import env_problem, golden, rel

F64, F32 = torch.float64, torch.float32
gpu = pytest.mark.gpu

DenseOut = namedtuple("DenseOut", "dC dc dtheta w AT rho cond")


# ------------------------------------------------------------------ the dense oracle
def _mt_pieces(port, x_init, C, c, x, u, dynamics, ns, nc, lo, hi):
    T = x.shape[0]
    F, f = port.linearize_dynamics(x, u, dynamics)
    cb = port.c_back(C, c, x, u)
    Ks, _, _ = port.lqr_backward(C, cb, F, None, u, ns, nc, lo, hi)
    Ks = torch.stack(Ks, 0)                              # reverse-time stack (:617-618)
    grad_D, grad_d, Dx, Du, _, d_x, d_u = port.grad_input(dynamics, x, u, Ks)
    return dict(T=T, F=F, f=f, grad_D=grad_D, grad_d=grad_d, Dx=Dx, Du=Du, d_x=d_x, d_u=d_u)


def _apply_mt(port, P, w, x_init, C, c, x, u, ns, nc, lo, hi):
    """M'w of port.dilqr_backward (one KKT pass + the contraction), any batch."""
    T = P["T"]
    k = port.kkt_backward(w[:, :, :ns], w[:, :, ns:], x_init, C, c, P["F"], P["f"], x, u, ns, nc,
                          lo, hi, gain_solve="chol_reg")
    Mw = torch.zeros_like(w)
    Mw[:T - 1, :, :ns] = torch.einsum("tbnm,tbnmk->tbk", k.dF, P["Dx"]) + \
        torch.einsum("tbn,tbnk->tbk", k.df, P["d_x"])
    Mw[:T - 1, :, ns:] = torch.einsum("tbnm,tbnmk->tbk", k.dF, P["Du"]) + \
        torch.einsum("tbn,tbnk->tbk", k.df, P["d_u"])
    return Mw, k


def _rep(t, L, dim=1):
    if t is None or not torch.is_tensor(t) or t.dim() == 0:
        return t
    reps = [1] * t.dim()
    reps[dim] = L
    return t.repeat(*reps)


def dense_mt(port, x_init, C, c, x, u, dynamics, ns, nc, lo=None, hi=None):
    """(M'_b [B, L, L] with L = T n, pieces): column e of M'_b is M' applied to the unit vector
    e; all L unit vectors go through one batched KKT pass (problem e B + b is b's copy)."""
    T, B = x.shape[0], x.shape[1]
    n = ns + nc
    L = T * n
    P = _mt_pieces(port, x_init, C, c, x, u, dynamics, ns, nc, lo, hi)
    W = torch.zeros(T, L * B, n, dtype=x.dtype)
    for e in range(L):
        W[e // n, e * B:(e + 1) * B, e % n] = 1.0
    PR = dict(P, F=_rep(P["F"], L), f=_rep(P["f"], L), Dx=_rep(P["Dx"], L), Du=_rep(P["Du"], L),
              d_x=_rep(P["d_x"], L), d_u=_rep(P["d_u"], L))
    Mw, _ = _apply_mt(port, PR, W, _rep(x_init, L, 0), _rep(C, L), _rep(c, L), _rep(x, L),
                      _rep(u, L), ns, nc, _rep(lo, L), _rep(hi, L))
    MT = Mw.reshape(T, L, B, n).permute(2, 0, 3, 1).reshape(B, L, L)
    return MT, P


def flat(v):
    """[T,B,n] -> [B, T n] (the index t n + k of A')."""
    return v.permute(1, 0, 2).reshape(v.shape[1], -1)


def dilqr_backward_dense(dl_dx, dl_du, x_init, C, c, x, u, dynamics, n_state, n_ctrl,
                         u_lower=None, u_upper=None, port=None):
    """The reference's dense solve of A'w = g (fix_point_equ), then the final KKT pass and the
    dtheta contraction of port.dilqr_backward.  Also returns w, the dense A' and, per problem,
    rho(M) and cond(A)."""
    ns, nc = n_state, n_ctrl
    T, B = x.shape[0], x.shape[1]
    MT, P = dense_mt(port, x_init, C, c, x, u, dynamics, ns, nc, u_lower, u_upper)
    L = MT.shape[-1]
    AT = torch.eye(L, dtype=x.dtype) - MT
    g = torch.cat((dl_dx, dl_du), 2)
    wf = torch.linalg.solve(AT, flat(g).unsqueeze(-1)).squeeze(-1)
    w = wf.reshape(B, T, ns + nc).permute(1, 0, 2).contiguous()
    k = port.kkt_backward(w[:, :, :ns], w[:, :, ns:], x_init, C, c, P["F"], P["f"], x, u, ns, nc,
                          u_lower, u_upper, gain_solve="chol_reg")
    dtheta = torch.einsum("tbnm,tbnmk->bk", k.dF, P["grad_D"]) + \
        torch.einsum("tbn,tbnk->bk", k.df, P["grad_d"])
    rho = torch.linalg.eigvals(MT).abs().max(-1).values
    return DenseOut(k.dC, k.dc, dtheta, w, AT, rho, torch.linalg.cond(AT))


def backward_error(AT, g, w):
    """|g - A'w| / |g| per problem under the oracle's dense A'."""
    gf, wf = flat(g.double()), flat(w.double())
    r = gf - (AT @ wf.unsqueeze(-1)).squeeze(-1)
    return r.norm(dim=1) / gf.norm(dim=1)


def _mpc_kw(pdx, lqr_iter, eps=None):
    return dict(u_lower=pdx.lower, u_upper=pdx.upper, lqr_iter=lqr_iter,
                eps=pdx.mpc_eps if eps is None else eps, linesearch_decay=pdx.linesearch_decay,
                max_linesearch_iter=pdx.max_linesearch_iter)


# ------------------------------------------------------------------ CPU: the oracle
@pytest.mark.parametrize("env", ["pendulum", "cartpole", "cartpole_T50", "rocket"])
def test_dense_oracle_reproduces_reference(port, env):
    """dilqr_backward_dense == the reference's fix_point_equ (goldens) to 1e-10."""
    g = golden("ref_dilqr_%s.npz" % env)
    cls = {"pendulum": port.PendulumDx, "cartpole": port.CartpoleDx,
           "cartpole_T50": port.CartpoleDx, "rocket": port.RocketDx}[env]
    pdx = cls(params=g["theta"], dtype=F64)
    T, B = int(g["T"]), g["x0"].shape[0]
    C = torch.diag(g["q"])[None, None].repeat(T, B, 1, 1)
    c = g["p"][None, None].repeat(T, B, 1)
    extra = {"u_init": g["u_init"]} if "u_init" in g else {}
    o = port.mpc_forward(g["x0"], port.QuadCost(C, c), pdx, pdx.n_state, pdx.n_ctrl, T,
                         final_pass=False, **extra, **_mpc_kw(pdx, int(g["lqr_iter"]), eps=1e-9))
    d = dilqr_backward_dense(g["gx"], g["gu"], g["x0"], C, c, o.x, o.u, pdx, pdx.n_state,
                             pdx.n_ctrl, pdx.lower, pdx.upper, port=port)
    assert rel(d.dtheta.sum(0), g["dtheta"]) < 1e-10
    assert rel(d.dC, g["dC"]) < 1e-10
    assert rel(d.dc, g["dc"]) < 1e-10


# The hard case: cartpole near the benchmark's regime 2a (cold start, 10 iLQR iterations, so
# most problems are not at a fixed point), detach_unconverged=False.
HARD = dict(name="cartpole", T=30, B=8, sigma=0.5, seed=0, lqr_iter=10)


def _hard_problem(port, dtype=F64):
    h = HARD
    pdx, x0, C, c, kw = env_problem(port, h["name"], h["T"], h["B"], dtype, sigma=h["sigma"],
                                    seed=h["seed"])
    g = torch.Generator().manual_seed(7)
    gx = torch.randn(h["T"], h["B"], pdx.n_state, generator=g, dtype=F64).to(dtype)
    gu = torch.randn(h["T"], h["B"], pdx.n_ctrl, generator=g, dtype=F64).to(dtype)
    return pdx, x0, C, c, kw, gx, gu


def test_hard_case_is_beyond_richardson(port):
    """On the oracle's own solution of HARD: rho(M_b) > 1 for at least one problem, and 30
    Richardson passes leave a relative update above 1e-2."""
    pdx, x0, C, c, kw, gx, gu = _hard_problem(port)
    h = HARD
    o = port.mpc_forward(x0, port.QuadCost(C, c), pdx, 5, 1, h["T"], final_pass=False,
                         **dict(kw, lqr_iter=h["lqr_iter"]))
    d = dilqr_backward_dense(gx, gu, x0, C, c, o.x, o.u, pdx, 5, 1, pdx.lower, pdx.upper,
                             port=port)
    print("\n[hard] rho(M_b) = %s" % [round(float(r), 3) for r in d.rho])
    assert float(d.rho.max()) > 1.0
    r = port.dilqr_backward(gx, gu, x0, C, c, o.x, o.u, pdx, 5, 1, pdx.lower, pdx.upper,
                            n_passes=30)
    print("[hard] relative update after 30 Richardson passes: %.2e" % r.resid)
    assert r.resid > 1e-2


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _mods():
    return (importlib.import_module("differentiable-ilqr_b200._solver"),
            importlib.import_module("differentiable-ilqr_b200.env_dx"),
            importlib.import_module("differentiable-ilqr_b200._lib"))


def _solve_hard(dilqr, dev, port, dtype=F64):
    """HARD on the device (mpc_explicit.MPC forward): (pdx, x0, C, c, gx, gu, x*, u*, dx)."""
    _, env, _ = _mods()
    pdx, x0, C, c, kw, gx, gu = _hard_problem(port, dtype)
    h = HARD
    m = dilqr.mpc_explicit.MPC(5, 1, h["T"], lqr_iter=h["lqr_iter"], verbose=-1,
                               exit_unconverged=False, detach_unconverged=False, n_batch=h["B"], **kw)
    dx = env.CartpoleDx(pdx.params.to(dev, dtype))
    x, u, _ = m(x0.to(dev), dilqr.QuadCost(C.to(dev), c.to(dev)), dx)
    return pdx, x0, C, c, gx, gu, x.detach(), u.detach(), dx


def _backward(dev, x0, C, c, gx, gu, x, u, dx, **kw):
    """_solver.dilqr_backward on the device (factored path, no preparation from a forward):
    (dC[T,B,n,n], dc[T,B,n], dtheta[B,nth], stats)."""
    solver, _, _ = _mods()
    stats = {}
    out = solver.dilqr_backward(None if gx is None else gx.to(dev), gu.to(dev), x0.to(dev),
                                C.to(dev), c.to(dev), x, u, dx, 5, 1, dx.lower, dx.upper,
                                stats=stats, **kw)
    return out + (stats,)


def test_gmres_sizes_from_the_abi(dilqr):
    """Workspace size of the ABI = (restart + 1) basis vectors + the per-problem FP64 data,
    computed from shapes (no device needed); restart beyond T n is rejected, and the cycle
    budget splits max_iter into cycles of at most `restart` steps."""
    import ctypes as C
    _, _, lib = _mods()
    L = lib.lib()
    k = lib.DilqrKrylov()
    k.n_state, k.n_ctrl, k.T, k.n_batch, k.dtype = 5, 1, 50, 65536, lib.F64
    k.restart, k.max_iter = 64, 150
    vec = 50 * 65536 * 6 * 8
    nb = L.dilqr_krylov_workspace_bytes(C.byref(k))
    assert 65 * vec <= nb < 65 * vec + (5 * 65 + 64 * 65 // 2 + 2) * 65536 * 8 + 4096
    assert [L.dilqr_krylov_cycle_steps(C.byref(k), i) for i in range(4)] == [64, 64, 22, 0]
    k.restart = 301
    assert L.dilqr_krylov_workspace_bytes(C.byref(k)) == 0


# path -> the converged case of test_dilqr_backward_paths it runs (each asserts its path)
CONVERGED = ["fused-cartpole-dense", "fused-pendulum-dense", "factored-cartpole-dense",
             "factored-pendulum-tn", "fused-cartpole-n", "fused-cartpole-tn", "fused-cartpole-tile",
             "factored-cartpole-tile", "fused-cartpole-gx-none", "generic-cartpole-bounds"]


def _device_case(dilqr, dev, port, c, dtype, **mpc_kw):
    """A case of test_dilqr_backward_paths solved and differentiated through mpc_explicit.MPC
    with the given backward options: (grads, last_backward, x, u, problem)."""
    bp = importlib.import_module("test_dilqr_backward_paths")
    _, env, _ = _mods()
    il = importlib.import_module("differentiable-ilqr_b200.il")
    P = bp._problem(port, c)
    pdx, x0, (Cin, cin), _, (lo, hi), kw = P
    ns, nc = pdx.n_state, pdx.n_ctrl
    if torch.is_tensor(lo):
        lo, hi = lo.to(dev, dtype), hi.to(dev, dtype)
    cls = {"cartpole": env.CartpoleDx, "pendulum": env.PendulumDx, "rocket": env.RocketDx}[c.name]
    theta = pdx.params.to(dev, dtype).requires_grad_()
    m = dilqr.mpc_explicit.MPC(ns, nc, c.T, u_lower=lo, u_upper=hi, lqr_iter=c.lqr_iter,
                               verbose=-1, exit_unconverged=False, detach_unconverged=False,
                               prepare_in_forward=c.prepare, solo=c.solo, n_batch=c.B, **mpc_kw,
                               **kw)
    a = Cin.to(dev, dtype).requires_grad_()
    b = cin.to(dev, dtype).requires_grad_()
    Cm, cv = il.tile_cost(a, b, c.T, c.B) if c.cost == "tile" else (a, b)
    x, u, _ = m(x0.to(dev, dtype), dilqr.QuadCost(Cm, cv), cls(theta))
    gx, gu = bp._upstream(c.T, c.B, ns, nc, dtype)
    loss = (u * gu.to(dev)).sum()
    if not c.gx_none:
        loss = loss + (x * gx.to(dev)).sum()
    loss.backward()
    return (tuple(t.grad.detach().cpu() for t in (a, b, theta)), m.last_backward,
            x.detach().cpu(), u.detach().cpu(), P)


@gpu
@pytest.mark.parametrize("key", CONVERGED)
def test_gmres_equals_richardson_at_converged_points(dilqr, port, dev, key):
    bp = importlib.import_module("test_dilqr_backward_paths")
    c = bp.CASES[key]
    with warnings.catch_warnings():
        warnings.simplefilter("error")           # GMRES must converge here: no warning
        gm, st, _, u, P = _device_case(dilqr, dev, port, c, F64, adjoint_solver="gmres",
                                       gmres_tol=1e-13)
    ri, st_r, _, _, _ = _device_case(dilqr, dev, port, c, F64, richardson_passes=80,
                                  richardson_tol=1e-14)
    pdx, _, _, _, bounds, _ = P
    bp._check_path(c, st, u, bounds, pdx)
    assert st["solver"] == "gmres" and st["gmres"].unconverged == 0
    assert (st["fused"], st["factored"]) == (st_r["fused"], st_r["factored"])
    errs = [rel(a, b) for a, b in zip(gm, ri)]
    print("\n[%s] gmres iters %s..%s rel(dC|dq) %.1e rel(dc|dp) %.1e rel(dtheta) %.1e"
          % (key, int(st["gmres"].iters.min()), int(st["gmres"].iters.max()), *errs))
    for name, e, r in zip(("dC", "dc", "dtheta"), errs, ri):
        assert float(r.abs().max()) > 0, name
        assert e < 1e-12, (key, name, e)


@gpu
def test_gmres_rocket_generic_path_matches_dense_solve(dilqr, port, dev):
    """Rocket (generic path: every M'v is a full adjoint LQR solve): GMRES == the dense solve at
    the device's x*, u* within 10 cond(A_b) 1e-15 + 1e-10.  Compared with the dense solve rather
    than with Richardson because on the 40-problem rocket case of test_dilqr_backward_paths
    Richardson run to 1e-14 diverges (rho(M) > 1 for some problem)."""
    bp = importlib.import_module("test_dilqr_backward_paths")
    c = bp.CASES["generic-rocket-dense-b4"]
    (dC, dc, dth), st, x, u, P = _device_case(dilqr, dev, port, c, F64, adjoint_solver="gmres")
    pdx, x0, _, (Cd, cd), (lo, hi), _ = P
    bp._check_path(c, st, u, (lo, hi), pdx)
    gx, gu = bp._upstream(c.T, c.B, pdx.n_state, pdx.n_ctrl, F64)
    d = dilqr_backward_dense(gx, gu, x0, Cd, cd, x, u, pdx, pdx.n_state, pdx.n_ctrl, lo, hi,
                             port=port)
    bound = 10 * float(d.cond.max()) * 1e-15 + 1e-10
    errs = [rel(dC, d.dC), rel(dc, d.dc), rel(dth, d.dtheta.sum(0))]
    print("\n[rocket] rho %s cond max %.1e rel %s (bound %.1e)" % (
        [round(float(r), 3) for r in d.rho], float(d.cond.max()), ["%.1e" % e for e in errs], bound))
    assert st["gmres"].unconverged == 0
    assert max(errs) <= bound, errs


@gpu
def test_gmres_hard_case_matches_dense_solve(dilqr, port, dev):
    """HARD, full GMRES (restart = T n): at the device's own x*, u* the oracle's dense A' gives
    the device's w a backward error <= 1e-11, and dC, dc, dtheta agree with the dense solve per
    problem within 10 cond(A_b) 1e-15 + 1e-10 (relative)."""
    pdx, x0, C, c, gx, gu, x, u, dx = _solve_hard(dilqr, dev, port)
    T, n = HARD["T"], 6
    dC, dc, dth, st = _backward(dev, x0, C, c, gx, gu, x, u, dx, solver="gmres",
                                gmres_restart=T * n, gmres_max_iter=4 * T * n)
    d = dilqr_backward_dense(gx, gu, x0, C, c, x.cpu(), u.cpu(), pdx, 5, 1, pdx.lower, pdx.upper,
                             port=port)
    print("\n[hard on device x*] rho %s cond %s iters %s" % (
        [round(float(r), 3) for r in d.rho], ["%.1e" % float(v) for v in d.cond],
        st["gmres"].iters.tolist()))
    assert float(d.rho.max()) > 1.0             # still beyond Richardson at the device's x*
    be = backward_error(d.AT, torch.cat((gx, gu), 2), st["gmres"].w.cpu())
    print("[hard] backward error %s" % ["%.1e" % float(v) for v in be])
    assert float(be.max()) <= 1e-11
    for b in range(HARD["B"]):
        bound = 10 * float(d.cond[b]) * 1e-15 + 1e-10
        for name, a, r in (("dC", dC[:, b], d.dC[:, b]), ("dc", dc[:, b], d.dc[:, b]),
                           ("dtheta", dth[b], d.dtheta[b])):
            assert rel(a, r) <= bound, (b, name, rel(a, r), bound)


@gpu
def test_gmres_zero_upstream_gives_exact_zeros(dilqr, port, dev):
    """Problems whose upstream gradient is 0 (masked) get exact zeros and no iterations, next to
    problems that iterate."""
    pdx, x0, C, c, gx, gu, x, u, dx = _solve_hard(dilqr, dev, port)
    zero = [1, 4]
    gx, gu = gx.clone(), gu.clone()
    gx[:, zero], gu[:, zero] = 0.0, 0.0
    dC, dc, dth, st = _backward(dev, x0, C, c, gx, gu, x, u, dx, solver="gmres",
                                gmres_restart=180, gmres_max_iter=720)
    it = st["gmres"].iters
    for b in zero:
        assert int(it[b]) == 0 and float(st["gmres"].resid[b]) == 0.0
        assert bool((dC[:, b] == 0).all()) and bool((dc[:, b] == 0).all())
        assert bool((dth[b] == 0).all())
    assert int(it.max()) > 0 and bool(torch.isfinite(dC).all()) and bool(torch.isfinite(dth).all())


@gpu
def test_gmres_short_budget_warns(dilqr, port, dev):
    pdx, x0, C, c, gx, gu, x, u, dx = _solve_hard(dilqr, dev, port)
    with pytest.warns(UserWarning, match="GMRES left"):
        _, _, _, st = _backward(dev, x0, C, c, gx, gu, x, u, dx, solver="gmres",
                                gmres_restart=4, gmres_max_iter=6)
    assert st["gmres"].unconverged > 0
    assert int(st["gmres"].iters.max()) == 6


@gpu
def test_gmres_non_convex_adjoint_raises(dilqr, port, dev):
    """The negative-weight case of test_dilqr_backward_paths (a non-convex adjoint QP, where
    Richardson falls back to the line-searching kernels): GMRES raises instead of iterating on
    a map that is not linear."""
    bp = importlib.import_module("test_dilqr_backward_paths")
    _, _, lib = _mods()
    with pytest.raises(lib.DilqrLibraryError, match="not linear"):
        _device_case(dilqr, dev, port, bp.CASES["fallback-cartpole"], F64, adjoint_solver="gmres")


@gpu
def test_gmres_production_batch_is_tiled_base(dilqr, port, dev):
    """A batch of 65541 problems, problem b = base problem b % 41 (the HARD family), reproduces
    the base's w, dC, dc, dtheta and per-problem iteration counts bit for bit (default restart,
    so the hard problems restart)."""
    _, env, _ = _mods()
    base, big = 41, 65541
    h = dict(HARD, B=base)
    pdx, x0, C, c, kw = env_problem(port, "cartpole", h["T"], base, F64, sigma=h["sigma"],
                                    seed=h["seed"])
    g = torch.Generator().manual_seed(7)
    gx = torch.randn(h["T"], base, 5, generator=g, dtype=F64)
    gu = torch.randn(h["T"], base, 1, generator=g, dtype=F64)
    m = dilqr.mpc_explicit.MPC(5, 1, h["T"], lqr_iter=h["lqr_iter"], verbose=-1,
                               exit_unconverged=False, detach_unconverged=False, n_batch=base, **kw)
    dx = env.CartpoleDx(pdx.params.to(dev))
    x, u, _ = m(x0.to(dev), dilqr.QuadCost(C.to(dev), c.to(dev)), dx)
    idx = torch.arange(big) % base
    out = {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # the budget may leave hard problems unconverged
        for name, sel in (("base", slice(None)), ("big", idx)):
            r = _backward(dev, x0[sel], C[:, sel], c[:, sel], gx[:, sel], gu[:, sel],
                          x.detach()[:, sel.to(dev) if torch.is_tensor(sel) else sel].contiguous(),
                          u.detach()[:, sel.to(dev) if torch.is_tensor(sel) else sel].contiguous(),
                          dx, solver="gmres")
            out[name] = r
    (bC, bc, bth, bs), (gC, gc, gth, gs) = out["base"], out["big"]
    assert torch.equal(gs["gmres"].iters, bs["gmres"].iters[idx])
    assert torch.equal(gs["gmres"].w, bs["gmres"].w[:, idx.to(dev)])
    assert torch.equal(gC, bC[:, idx.to(dev)]) and torch.equal(gc, bc[:, idx.to(dev)])
    assert torch.equal(gth, bth[idx.to(dev)])
    assert bs["gmres"].iters.unique().numel() > 1   # problems stopped at different steps


@gpu
def test_gmres_deferred_equals_immediate(dilqr, port, dev):
    """il.ImitationStep(adjoint_solver="gmres"): the deferred step (whole budget enqueued, no host
    read) equals the immediate one bit for bit."""
    _, env, _ = _mods()
    il = importlib.import_module("differentiable-ilqr_b200.il")
    T, B = 20, 41
    step = il.ImitationStep(env.CartpoleDx, T, 10, F64, dev, adjoint_solver="gmres")
    g = torch.Generator().manual_seed(5)
    r = (torch.rand(B, 4, generator=g, dtype=F64) * 2 - 1) * 0.5
    x0 = torch.stack((r[:, 0], r[:, 1], torch.cos(r[:, 2]), torch.sin(r[:, 2]), r[:, 3]), 1)
    uexp = torch.randn(T, B, 1, generator=g, dtype=F64).to(dev)
    q, p = [t.to(dev, F64) for t in env.CartpoleDx().get_true_obj()]
    res = step.prepare(x0.to(dev), q, p, torch.tensor((9.8, 1.0, 0.1, 0.5), dtype=F64, device=dev))
    outs = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for defer in (True, False):
            step.defer = defer
            outs.append(step.run_resident(res, uexp).clone())
    assert step.mpc.last_backward["solver"] == "gmres"
    assert torch.equal(outs[0], outs[1]), (outs[0] - outs[1]).abs().max()


@gpu
def test_gmres_module_solver_and_op_agree(dilqr, port, dev):
    """mpc_explicit.MPC(adjoint_solver="gmres") == _solver.dilqr_backward == the torch op with
    adjoint_solver="gmres", bit for bit on cartpole (factored path: no preparation in the
    forward, as the op has none)."""
    _, env, lib = _mods()
    ops = importlib.import_module("differentiable-ilqr_b200.torch_ops")
    ops.load()
    pdx, x0, C, c, gx, gu, x, u, dx = _solve_hard(dilqr, dev, port)
    h = HARD
    kw = dict(u_lower=pdx.lower, u_upper=pdx.upper, eps=pdx.mpc_eps,
              linesearch_decay=pdx.linesearch_decay, max_linesearch_iter=pdx.max_linesearch_iter)
    theta = pdx.params.to(dev, F64).requires_grad_()
    Cg, cg = C.to(dev).requires_grad_(), c.to(dev).requires_grad_()
    m = dilqr.mpc_explicit.MPC(5, 1, h["T"], lqr_iter=h["lqr_iter"], verbose=-1,
                               exit_unconverged=False, detach_unconverged=False, n_batch=h["B"],
                               adjoint_solver="gmres", prepare_in_forward=False, **kw)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        xm, um, _ = m(x0.to(dev), dilqr.QuadCost(Cg, cg), env.CartpoleDx(theta))
        ((xm * gx.to(dev)).sum() + (um * gu.to(dev)).sum()).backward()
        dC, dc, dth, st = _backward(dev, x0, C, c, gx, gu, xm.detach(), um.detach(), dx,
                                    solver="gmres")
        oC, oc, oth = torch.ops.dilqr.dilqr_backward(
            gx.to(dev), gu.to(dev), x0.to(dev), C.to(dev), c.to(dev), xm.detach(), um.detach(),
            pdx.params.to(dev), lib.DYN_CARTPOLE, pdx.lower, pdx.upper, 30,
            pdx.max_linesearch_iter, pdx.linesearch_decay, adjoint_solver="gmres")
    assert st["factored"] and not st["fused"] and m.last_backward["solver"] == "gmres"
    assert torch.equal(Cg.grad, dC) and torch.equal(cg.grad, dc)
    assert torch.equal(theta.grad, dth.sum(0))
    assert torch.equal(oC, dC) and torch.equal(oc, dc) and torch.equal(oth, dth)


@gpu
def test_gmres_fp32_at_a_converged_point(dilqr, port, dev):
    """FP32 at a converged point: backward error <= 1e-5 under the FP64 oracle's dense A', and
    dtheta within 10x of the FP32 oracle's own error against FP64."""
    _, env, _ = _mods()
    T, B = 20, 16
    pdx, x0, C, c, kw = env_problem(port, "cartpole", T, B, F64, sigma=0.05)
    kw["eps"] = 1e-9
    o = port.mpc_forward(x0, port.QuadCost(C, c), pdx, 5, 1, T, lqr_iter=60, final_pass=False,
                         **kw)
    g = torch.Generator().manual_seed(9)
    gx = torch.randn(T, B, 5, generator=g, dtype=F64)
    gu = torch.randn(T, B, 1, generator=g, dtype=F64)
    d = dilqr_backward_dense(gx, gu, x0, C, c, o.x, o.u, pdx, 5, 1, pdx.lower, pdx.upper,
                             port=port)
    dx32 = env.CartpoleDx(pdx.params.to(dev, F32))
    f = lambda t: t.to(dev, F32)                                     # noqa: E731
    _, _, dth, st = _backward(dev, f(x0), f(C), f(c), f(gx), f(gu), f(o.x), f(o.u), dx32,
                              solver="gmres")
    be = backward_error(d.AT, torch.cat((gx, gu), 2).float(), st["gmres"].w.cpu())
    p32 = port.CartpoleDx(params=pdx.params.float(), dtype=F32)
    r32 = port.dilqr_backward(gx.float(), gu.float(), x0.float(), C.float(), c.float(),
                              o.x.float(), o.u.float(), p32, 5, 1, p32.lower, p32.upper,
                              n_passes=30, tol=1e-7)
    e_dev, e_ora = rel(dth.sum(0), d.dtheta.sum(0)), rel(r32.dtheta.sum(0), d.dtheta.sum(0))
    print("\n[fp32] backward error %.1e, dtheta err device %.1e oracle(fp32) %.1e"
          % (float(be.max()), e_dev, e_ora))
    assert float(be.max()) <= 1e-5
    assert e_dev <= 10 * e_ora
