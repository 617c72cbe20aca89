"""The DiLQR backward (`_solver.dilqr_backward`) on each of its four paths against the CPU
oracle (`port.dilqr_backward`), run on the device's own forward solution.

The forward solve runs on the device; its x*, u* and every input of the backward (upstream
gradient, bounds, cost, theta) are then handed to the oracle unchanged, with the same number
of Richardson passes.  The forward's amplification of last-bit differences therefore plays no
part and only the backward is measured: dC, dc, dtheta (and dq, dp of `il.tile_cost`) hold
1e-9 relative in FP64.

The four paths (`m.last_backward["fused"]` / `["factored"]`):
- fused: pendulum / cartpole, scalar bounds, n_ctrl = 1, preparation enqueued by the forward;
- factored: the same models with `prepare_in_forward=False`;
- generic: rocket, or tensor `u_lower` / `u_upper`;
- fallback: the factored passes found an adjoint step the reference's line search rejects
  (a non-convex adjoint QP); the backward is recomputed on the generic path.
Every GPU case asserts the path it took, from the table `CASES` written out by hand, so a
change of routing fails here instead of moving the coverage elsewhere.

FP32 (one case per path): the device's FP32 gradient is compared with the oracle run in FP32
on the same inputs, both measured against the oracle in FP64.  A kernel error then shows up
as an error far beyond what an FP32 implementation of the same algorithm makes, whatever the
conditioning of the problem.

The CPU tests at the end show on the oracle that each feature a case is about (asymmetric C,
tensor bounds, the negative weight of the fallback case) moves the gradient by more than 100x
the FP64 bound, so a device that ignored it would fail."""
import importlib
import time
from collections import namedtuple

import pytest
import torch

from common import env_problem, rel

F64, F32 = torch.float64, torch.float32
TOL = 1e-9                 # FP64 bound on dC, dc, dtheta, dq, dp
GX_SEED = 11
gpu = pytest.mark.gpu

# path -> (last_backward["fused"], last_backward["factored"])
PATH_FLAGS = {"fused": (True, True), "factored": (False, True), "generic": (False, False),
              "fallback": (False, False)}

Case = namedtuple("Case", "path name T B cost bounds sigma seed lqr_iter passes tol prepare solo "
                          "gx_none qneg")


def case(path, name, T, B, cost="dense", bounds="scalar", sigma=0.3, seed=0, lqr_iter=40,
         passes=30, tol=None, prepare=True, solo=False, gx_none=False, qneg=None):
    """``tol``: None = fixed pass count; "default" = MPC's richardson_tol (1e-14)."""
    return Case(path, name, T, B, cost, bounds, sigma, seed, lqr_iter, passes, tol, prepare, solo,
                gx_none, qneg)


# cost: "dense" C[T,B,n,n]; "n" C[n,n]; "tn" C[T,n,n]; "asym" dense with C != C';
# "tile" il.tile_cost(q, p, T, B).  bounds: "scalar" (the model's box) or "tensor" [T,B,1].
CASES = {
    # ---- fused
    "fused-cartpole-dense": case("fused", "cartpole", 20, 70),
    "fused-cartpole-n": case("fused", "cartpole", 16, 33, cost="n"),
    "fused-cartpole-tn": case("fused", "cartpole", 16, 45, cost="tn"),
    "fused-cartpole-asym": case("fused", "cartpole", 16, 40, cost="asym"),
    "fused-cartpole-tile": case("fused", "cartpole", 20, 45, cost="tile"),
    "fused-cartpole-gx-none": case("fused", "cartpole", 16, 37, gx_none=True),
    "fused-cartpole-tol": case("fused", "cartpole", 16, 40, tol="default", passes=80),
    "fused-pendulum-dense": case("fused", "pendulum", 20, 64, sigma=0.5),
    "fused-pendulum-n": case("fused", "pendulum", 16, 33, cost="n", sigma=0.5),
    "fused-pendulum-tn": case("fused", "pendulum", 16, 40, cost="tn", sigma=0.5),
    "fused-pendulum-asym": case("fused", "pendulum", 16, 45, cost="asym", sigma=0.5),
    "fused-pendulum-tile": case("fused", "pendulum", 16, 50, cost="tile", sigma=0.5),
    "fused-pendulum-gx-none": case("fused", "pendulum", 16, 33, gx_none=True, sigma=0.5),
    "fused-pendulum-tol": case("fused", "pendulum", 16, 40, tol="default", passes=80, sigma=0.5),
    "fused-pendulum-solo1": case("fused", "pendulum", 20, 45, sigma=1.0, lqr_iter=100, solo=True),
    "fused-pendulum-solo2": case("fused", "pendulum", 20, 45, sigma=1.0, lqr_iter=100, solo=2),
    # ---- factored (no preparation in the forward)
    "factored-cartpole-dense": case("factored", "cartpole", 20, 70, prepare=False),
    "factored-cartpole-n": case("factored", "cartpole", 16, 33, cost="n", prepare=False),
    "factored-cartpole-asym": case("factored", "cartpole", 16, 40, cost="asym", prepare=False),
    "factored-cartpole-tile": case("factored", "cartpole", 20, 45, cost="tile", prepare=False),
    "factored-cartpole-gx-none": case("factored", "cartpole", 16, 37, gx_none=True,
                                      prepare=False),
    "factored-pendulum-tn": case("factored", "pendulum", 16, 40, cost="tn", sigma=0.5,
                                 prepare=False),
    "factored-pendulum-tile": case("factored", "pendulum", 16, 50, cost="tile", sigma=0.5,
                                   prepare=False),
    "factored-pendulum-tol": case("factored", "pendulum", 16, 40, tol="default", passes=80,
                                  sigma=0.5, prepare=False),
    "factored-pendulum-solo1": case("factored", "pendulum", 20, 45, sigma=1.0, lqr_iter=100,
                                    solo=True, prepare=False),
    # ---- generic
    "generic-rocket-dense-b4": case("generic", "rocket", 10, 4, lqr_iter=20, passes=20),
    "generic-rocket-dense": case("generic", "rocket", 10, 40, lqr_iter=20, passes=20),
    "generic-rocket-n": case("generic", "rocket", 10, 40, cost="n", lqr_iter=20, passes=20),
    "generic-rocket-tn": case("generic", "rocket", 10, 37, cost="tn", lqr_iter=20, passes=20),
    "generic-rocket-tile": case("generic", "rocket", 10, 40, cost="tile", lqr_iter=20,
                                passes=20),
    "generic-cartpole-bounds": case("generic", "cartpole", 16, 45, bounds="tensor"),
    "generic-pendulum-bounds": case("generic", "pendulum", 16, 45, bounds="tensor", sigma=1.0),
    "generic-pendulum-bounds-n": case("generic", "pendulum", 16, 40, cost="n", bounds="tensor",
                                      sigma=1.0),
    "generic-cartpole-bounds-tol": case("generic", "cartpole", 12, 33, bounds="tensor",
                                        tol="default", passes=80),
    # ---- fallback: a negative weight on the pole's angular velocity in every third problem
    # (in all of them for the broadcast C[T,n,n]) makes their adjoint QP non-convex (see
    # test_fallback_problem_is_non_convex)
    "fallback-cartpole": case("fallback", "cartpole", 8, 45, qneg=-1.0, passes=10),
    "fallback-cartpole-tn": case("fallback", "cartpole", 8, 40, cost="tn", qneg=-1.0, passes=10),
}

F32_CASES = ["fused-cartpole-dense", "factored-pendulum-tn", "generic-rocket-dense",
             "generic-cartpole-bounds", "fused-cartpole-tile"]


def _neg_rows(B):
    return torch.arange(B) % 3 == 0


def _bounds(port, c, pdx):
    """Scalar box, or [T,B,1] bounds per problem: a third keep the box, the others are
    tightened (differently above and below, and slightly over time) so that the active sets
    differ between problems."""
    if c.bounds == "scalar":
        return pdx.lower, pdx.upper
    g = torch.Generator().manual_seed(31 + c.seed)
    # the box's fraction per problem: the pendulum saturates +-2 often, the cartpole's
    # forces (|u| < 25 here) are far inside +-100
    s = torch.tensor((1.0, 0.5, 0.15) if c.name == "pendulum" else (1.0, 0.08, 0.03), dtype=F64)
    up = s[torch.randint(0, 3, (c.B,), generator=g)]
    lo = s[torch.randint(0, 3, (c.B,), generator=g)]
    ramp = 1.0 + 0.1 * torch.linspace(0, 1, c.T, dtype=F64)[:, None]
    up = torch.where(up < 1, up * ramp, up)        # [T,B]
    lo = torch.where(lo < 1, lo * ramp, lo)
    return (pdx.lower * lo)[..., None].contiguous(), (pdx.upper * up)[..., None].contiguous()


def _problem(port, c):
    """The case's inputs in FP64 on the CPU: (pdx, x0, cost handed to the device, its dense
    [T,B,..] form for the oracle, bounds, solver keywords)."""
    pdx, x0, C, cv, kw = env_problem(port, c.name, c.T, c.B, F64, sigma=c.sigma, seed=c.seed)
    kw["eps"] = 1e-9
    del kw["u_lower"], kw["u_upper"]
    n = C.shape[-1]
    C, cv = C.clone(), cv.clone()
    if c.qneg is not None:
        iw = {"pendulum": 2, "cartpole": 4}[c.name]
        C[:, _neg_rows(c.B), iw, iw] = c.qneg
    if c.cost == "asym":          # test_gpu_parity.test_asymmetric_cost_uses_dense_path
        g = torch.Generator().manual_seed(21)
        skew = torch.randn(c.T, c.B, n, n, generator=g, dtype=F64) * 1e-3
        skew[:, :, -1, :] = 0.0
        skew[:, :, :, -1] = 0.0
        C = C + torch.triu(skew, 1)
    ramp = 1.0 + 0.5 * torch.linspace(0, 1, c.T, dtype=F64)
    if c.cost == "n":
        Cin, cin = C[0, 0].clone(), cv[0, 0].clone()
    elif c.cost == "tn":          # a time-varying C[T,n,n] (with the negative weight if any)
        Cin, cin = C[:, 0] * ramp[:, None, None], cv[:, 0] * ramp[:, None]
    else:
        Cin, cin = C, cv
    if c.cost == "tile":
        q, p = pdx.get_true_obj()
        Cin, cin = q.clone(), p.clone()
        Cd, cd = torch.diag(q)[None, None].expand(c.T, c.B, n, n), p[None, None].expand(c.T, c.B, n)
    else:
        Cd = Cin.expand(c.T, c.B, n, n) if Cin.dim() == 2 else (
            Cin[:, None].expand(c.T, c.B, n, n) if Cin.dim() == 3 else Cin)
        cd = cin.expand(c.T, c.B, n) if cin.dim() == 1 else (
            cin[:, None].expand(c.T, c.B, n) if cin.dim() == 2 else cin)
    lo, hi = _bounds(port, c, pdx)
    return pdx, x0, (Cin, cin), (Cd.contiguous(), cd.contiguous()), (lo, hi), kw


def _upstream(T, B, ns, nc, dtype):
    g = torch.Generator().manual_seed(GX_SEED)
    gx = torch.randn(T, B, ns, generator=g, dtype=F64).to(dtype)
    gu = torch.randn(T, B, nc, generator=g, dtype=F64).to(dtype)
    return gx, gu


def _oracle(port, c, pdx, x0, dense, bounds, x, u, gx, gu, dtype):
    """port.dilqr_backward in ``dtype`` on the device's solution (x, u), reduced to the
    layout of the cost the device was handed: (dC, dc, dtheta) or (dq, dp, dtheta)."""
    cls = type(pdx)
    od = cls(params=pdx.params.to(dtype), dtype=dtype)
    lo, hi = bounds
    if torch.is_tensor(lo):
        lo, hi = lo.to(dtype), hi.to(dtype)
    Cd, cd = dense[0].to(dtype), dense[1].to(dtype)
    x, u, gu = x.to(dtype), u.to(dtype), gu.to(dtype)
    gx = torch.zeros_like(x) if gx is None else gx.to(dtype)
    n_passes, tol = (c.passes, None) if c.tol is None else (60, 1e-15)
    o = port.dilqr_backward(gx, gu, x0.to(dtype), Cd, cd, x, u, od, od.n_state, od.n_ctrl, lo, hi,
                            n_passes=n_passes, tol=tol)
    dC, dc = o.dC, o.dc
    if c.cost == "tile":
        dC, dc = dC.diagonal(dim1=-2, dim2=-1).sum((0, 1)), dc.sum((0, 1))
    elif c.cost == "n":
        dC, dc = dC.sum((0, 1)), dc.sum((0, 1))
    elif c.cost == "tn":
        dC, dc = dC.sum(1), dc.sum(1)
    return dC, dc, o.dtheta.sum(0)


def _device(dilqr, dev, port, c, dtype):
    """Solve and differentiate on the device through mpc_explicit.MPC.  Returns
    (x, u, gx, gu, (dC | dq, dc | dp, dtheta), last_backward, problem)."""
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    il = importlib.import_module("differentiable-ilqr_b200.il")
    P = _problem(port, c)
    pdx, x0, (Cin, cin), _, (lo, hi), kw = P
    ns, nc = pdx.n_state, pdx.n_ctrl
    if torch.is_tensor(lo):
        lo, hi = lo.to(dev, dtype), hi.to(dev, dtype)
    cls = {"cartpole": env.CartpoleDx, "pendulum": env.PendulumDx, "rocket": env.RocketDx}[c.name]
    theta = pdx.params.to(dev, dtype).requires_grad_()
    extra = {} if c.tol == "default" else {"richardson_tol": None}
    m = dilqr.mpc_explicit.MPC(ns, nc, c.T, u_lower=lo, u_upper=hi, lqr_iter=c.lqr_iter,
                               verbose=-1, exit_unconverged=False, detach_unconverged=False,
                               richardson_passes=c.passes, prepare_in_forward=c.prepare,
                               solo=c.solo, n_batch=c.B, **extra, **kw)
    a = Cin.to(dev, dtype).requires_grad_()
    b = cin.to(dev, dtype).requires_grad_()
    C, cv = il.tile_cost(a, b, c.T, c.B) if c.cost == "tile" else (a, b)
    x, u, _ = m(x0.to(dev, dtype), dilqr.QuadCost(C, cv), cls(theta))
    gx, gu = _upstream(c.T, c.B, ns, nc, dtype)
    loss = (u * gu.to(dev)).sum()
    if not c.gx_none:
        loss = loss + (x * gx.to(dev)).sum()
    loss.backward()
    grads = tuple(t.grad.detach().cpu() for t in (a, b, theta))
    return (x.detach().cpu(), u.detach().cpu(), None if c.gx_none else gx, gu, grads,
            m.last_backward, P)


def _active(u, lo, hi):
    return (torch.abs(u - lo) <= 1e-8) | (torch.abs(u - hi) <= 1e-8)


def _check_path(c, stats, u, bounds, pdx):
    fused, factored = PATH_FLAGS[c.path]
    assert stats["fused"] is fused and stats["factored"] is factored, (c.path, stats)
    if c.path in ("fused", "factored", "fallback"):
        assert c.name != "rocket" and not torch.is_tensor(bounds[0])
    if c.tol == "default":
        assert stats["passes"] < c.passes, stats          # richardson_tol stopped the loop
    if c.bounds == "tensor":
        lo, hi = bounds
        act = _active(u, lo.to(u.dtype), hi.to(u.dtype))
        tight = (hi < pdx.upper) | (lo > pdx.lower)
        assert bool((act & tight).any()), "no tightened bound active"
        assert act.sum((0, 2)).unique().numel() > 1       # active sets differ between problems


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@gpu
@pytest.mark.parametrize("key", list(CASES))
def test_backward_vs_oracle_f64(dilqr, port, dev, key):
    c = CASES[key]
    x, u, gx, gu, grads, stats, P = _device(dilqr, dev, port, c, F64)
    pdx, x0, _, dense, bounds, _ = P
    _check_path(c, stats, u, bounds, pdx)
    t0 = time.time()
    ref = _oracle(port, c, pdx, x0, dense, bounds, x, u, gx, gu, F64)
    errs = [rel(a, b) for a, b in zip(grads, ref)]
    print("\n[%s] path=%s passes=%s rel(dC|dq)=%.1e rel(dc|dp)=%.1e rel(dtheta)=%.1e oracle %.1fs"
          % (key, c.path, stats["passes"], *errs, time.time() - t0))
    for name, e, r in zip(("dC", "dc", "dtheta"), errs, ref):
        assert float(r.abs().max()) > 0, name
        assert e < TOL, (key, name, e)


@gpu
@pytest.mark.parametrize("key", F32_CASES)
def test_backward_vs_oracle_f32(dilqr, port, dev, key):
    """rel(device32, oracle64) <= 10 rel(oracle32, oracle64) (floor 1e-5), with
    rel(oracle32, oracle64) < 1e-2 so that the yardstick means something."""
    c = CASES[key]
    x, u, gx, gu, grads, stats, P = _device(dilqr, dev, port, c, F32)
    pdx, x0, _, dense, bounds, _ = P
    # both oracle runs start from the FP32 inputs the device was handed
    r32 = lambda t: t.to(F32) if torch.is_tensor(t) else t
    pdx = type(pdx)(params=pdx.params.to(F32), dtype=F32)
    x0, dense, bounds = x0.to(F32), tuple(map(r32, dense)), tuple(map(r32, bounds))
    _check_path(c, stats, u, bounds, pdx)
    o32 = _oracle(port, c, pdx, x0, dense, bounds, x, u, gx, gu, F32)
    o64 = _oracle(port, c, pdx, x0, dense, bounds, x, u, gx, gu, F64)
    for name, d, a, b in zip(("dC", "dc", "dtheta"), grads, o32, o64):
        yard = rel(a, b)
        err = rel(d, b)
        print("\n[%s f32] %s rel(dev32, o64)=%.1e rel(o32, o64)=%.1e" % (key, name, err, yard))
        assert yard < 1e-2, (key, name, yard)
        assert err <= max(10 * yard, 1e-5), (key, name, err, yard)


@gpu
def test_fallback_through_imitation_step(dilqr, port, dev):
    """il.ImitationStep defers the adjoint line-search check to the end of the step; with a
    negative weight on the pole's angular velocity the check fails, the step is repeated with
    immediate checks (``redone`` + 1), whose backward falls back to the generic path.  Its
    (dtheta, dq, dp) match the oracle at the step's own solution."""
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    il = importlib.import_module("differentiable-ilqr_b200.il")
    T, B, n_rich = 8, 45, 4
    c = case("fallback", "cartpole", T, B, cost="tile", qneg=-1.0, passes=n_rich)
    pdx, x0, (q, p), _, _, _ = _problem(port, c)
    q = q.clone()
    q[4] = -1.0
    g = torch.Generator().manual_seed(5)
    uexp = torch.randn(T, B, 1, generator=g, dtype=F64).to(dev)
    step = il.ImitationStep(env.CartpoleDx, T=T, lqr_iter=20, dtype=F64, device=dev,
                            n_richardson=n_rich)
    seen = []
    step.mpc.register_forward_hook(lambda mod, inp, out: seen.append(out))
    res = step.prepare(x0.to(dev), q.to(dev), p.to(dev), pdx.params.to(dev))
    flat = step.run_resident(res, uexp).cpu()
    assert step.redone == 1
    assert step.mpc.last_backward["factored"] is False and step.mpc.last_backward["fused"] is False
    x, u = seen[-1][0].detach().cpu(), seen[-1][1].detach().cpu()
    gu = 2.0 * (u - uexp.cpu()) / u.numel()
    n = q.shape[0]
    dense = (torch.diag(q)[None, None].expand(T, B, n, n).contiguous(),
             p[None, None].expand(T, B, n).contiguous())
    dq, dp, dth = _oracle(port, c, pdx, x0, dense, (pdx.lower, pdx.upper), x, u, None, gu, F64)
    nth = pdx.params.numel()
    for name, d, r in (("dtheta", flat[:nth], dth), ("dq", flat[nth:nth + n], dq),
                       ("dp", flat[nth + n:nth + 2 * n], dp)):
        print("\n[imitation fallback] %s rel=%.1e" % (name, rel(d, r)))
        assert rel(d, r) < TOL, (name, rel(d, r))


# ------------------------------------------------------------------ non-vacuity (CPU)
def _oracle_at_own_solution(port, c, mutate=None):
    pdx, x0, _, dense, bounds, kw = _problem(port, c)
    if mutate is not None:
        dense, bounds = mutate(dense, bounds)
    o = port.mpc_forward(x0, port.QuadCost(*dense), pdx, pdx.n_state, pdx.n_ctrl, c.T,
                         u_lower=bounds[0], u_upper=bounds[1], lqr_iter=c.lqr_iter,
                         final_pass=False, **kw)
    gx, gu = _upstream(c.T, c.B, pdx.n_state, pdx.n_ctrl, F64)
    return pdx, x0, dense, bounds, o, gx, gu


def _shift(port, c, mutate):
    """max over (dC, dc, dtheta) of rel(oracle with the feature, oracle without it), both at
    the solution of the problem with the feature (the device's inputs in the GPU test)."""
    pdx, x0, dense, bounds, o, gx, gu = _oracle_at_own_solution(port, c)
    a = _oracle(port, c, pdx, x0, dense, bounds, o.x, o.u, gx, gu, F64)
    dense2, bounds2 = mutate(dense, bounds)
    b = _oracle(port, c, pdx, x0, dense2, bounds2, o.x, o.u, gx, gu, F64)
    return max(rel(x, y) for x, y in zip(a, b))


def test_asymmetric_cost_changes_oracle_result(port):
    c = CASES["fused-cartpole-asym"]
    d = _shift(port, c, lambda D, bd: ((0.5 * (D[0] + D[0].transpose(-1, -2)), D[1]), bd))
    assert d > 100 * TOL, d


def test_tensor_bounds_change_oracle_result(port):
    for key in ("generic-pendulum-bounds", "generic-cartpole-bounds"):
        c = CASES[key]
        pdx = {"pendulum": port.PendulumDx, "cartpole": port.CartpoleDx}[c.name]
        d = _shift(port, c, lambda D, bd: (D, (pdx.lower, pdx.upper)))
        assert d > 100 * TOL, (key, d)


def test_fallback_weight_changes_oracle_result(port):
    c = CASES["fallback-cartpole"]

    def zero(D, bd):
        C = D[0].clone()
        C[:, _neg_rows(c.B), 4, 4] = 0.0
        return (C, D[1]), bd
    assert _shift(port, c, zero) > 100 * TOL


def test_fallback_problem_is_non_convex(port):
    """The fallback cases' adjoint QP is not convex for some problems: the reference's line
    search (port.lqr_step on the adjoint LQR of the first Richardson pass) rejects the full
    step there, and (dense cost) in no problem without the negative weight."""
    for key in ("fallback-cartpole", "fallback-cartpole-tn"):
        c = CASES[key]
        pdx, x0, dense, bounds, o, gx, gu = _oracle_at_own_solution(port, c)
        F, _ = port.linearize_dynamics(o.x, o.u, pdx)
        r = torch.cat((gx, gu), 2)
        I = _active(o.u, *bounds)
        zero = torch.zeros_like(x0)
        u0 = torch.zeros_like(o.u)
        lin = port.LinDx(F, None)
        s = port.lqr_step(zero, dense[0], -r, F, port.get_traj(c.T, u0, zero, lin), u0,
                          port.QuadCost(dense[0], -r), lin, pdx.n_state, pdx.n_ctrl, u_zero_I=I,
                          gain_solve="chol_reg")
        rejected = s.alphas < 1
        assert bool(rejected.any()), key
        shared = c.cost in ("n", "tn")      # a broadcast cost carries the weight everywhere
        assert shared or not bool((rejected & ~_neg_rows(c.B)).any()), key
