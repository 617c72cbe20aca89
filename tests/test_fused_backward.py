"""GPU tests of the fused DiLQR backward (round 2): the one-sweep gains + costates
kernel, the (t, problem)-parallel second-order tables, the adjoint passes on the split
upstream gradient, the in-kernel reduction to the gradient of the tiled cost, and the
deferred validation reads -- each against the round-1 kernel sequence (itself pinned to
the reference's goldens in test_gpu_parity.py) and against the oracle."""
import importlib

import pytest
import torch

from common import env_problem, rel

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def env():
    return importlib.import_module("differentiable-ilqr_b200.env_dx")


def _solve_and_grad(dilqr, env, dev, name, T, B, port, fused, passes=40, sigma=0.05, seed=0,
                    lqr_iter=60, gx_none=False):
    solver = importlib.import_module("differentiable-ilqr_b200._solver")
    pdx, x0, C, c, kw = env_problem(port, name, T, B, torch.float64, sigma=sigma, seed=seed)
    kw["eps"] = 1e-9
    cls = {"cartpole": env.CartpoleDx, "pendulum": env.PendulumDx}[name]
    theta = pdx.params.to(dev).requires_grad_()
    Cg, cg = C.to(dev).requires_grad_(), c.to(dev).requires_grad_()
    m = dilqr.mpc_explicit.MPC(pdx.n_state, pdx.n_ctrl, T, lqr_iter=lqr_iter, verbose=-1,
                               exit_unconverged=False, detach_unconverged=False,
                               richardson_passes=passes, richardson_tol=None, **kw)
    old = solver.FUSED_BACKWARD
    solver.FUSED_BACKWARD = fused
    try:
        x, u, _ = m(x0.to(dev), dilqr.QuadCost(Cg, cg), cls(theta))
        g = torch.Generator().manual_seed(11)
        gx = torch.randn(x.shape, generator=g, dtype=torch.float64).to(dev)
        gu = torch.randn(u.shape, generator=g, dtype=torch.float64).to(dev)
        loss = (u * gu).sum() if gx_none else (x * gx).sum() + (u * gu).sum()
        loss.backward()
    finally:
        solver.FUSED_BACKWARD = old
    assert m.last_backward["fused"] == fused
    return x.detach(), u.detach(), theta.grad, Cg.grad, cg.grad


@pytest.mark.parametrize("name,T,B,sigma", [("cartpole", 50, 96, 0.05), ("cartpole", 20, 70, 0.3),
                                            ("pendulum", 20, 64, 1.0), ("pendulum", 12, 33, 0.5)])
def test_fused_equals_round1_sequence(dilqr, port, env, dev, name, T, B, sigma):
    """Same solve, same upstream gradient: the fused kernels reproduce the round-1 sequence
    (whose outputs are pinned to the reference's dense fix_point_equ) to rounding."""
    a = _solve_and_grad(dilqr, env, dev, name, T, B, port, True, sigma=sigma)
    b = _solve_and_grad(dilqr, env, dev, name, T, B, port, False, sigma=sigma)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for i in (2, 3, 4):
        assert rel(a[i], b[i]) < 1e-12, (i, rel(a[i], b[i]))


def test_fused_no_state_gradient(dilqr, port, env, dev):
    """dl/dx = None (imitation loss on the controls only): the kernels read a null gx."""
    a = _solve_and_grad(dilqr, env, dev, "cartpole", 30, 64, port, True, gx_none=True)
    b = _solve_and_grad(dilqr, env, dev, "cartpole", 30, 64, port, False, gx_none=True)
    for i in (2, 3, 4):
        assert rel(a[i], b[i]) < 1e-12


def test_fused_pendulum_active_constraints(dilqr, port, env, dev):
    """Pendulum swing-up saturates the torque bound: pnqp in the gains sweep (trace replay)
    and the active-set mask in the factor / passes."""
    a = _solve_and_grad(dilqr, env, dev, "pendulum", 20, 64, port, True, sigma=1.0, lqr_iter=100)
    u = a[1]
    assert float(((u.abs() - 2.0).abs() < 1e-8).float().mean()) > 0.01   # some controls at +-2
    o = _solve_and_grad(dilqr, env, dev, "pendulum", 20, 64, port, False, sigma=1.0, lqr_iter=100)
    for i in (2, 3, 4):
        assert rel(a[i], o[i]) < 1e-12


@pytest.mark.parametrize("name", ["cartpole", "pendulum"])
def test_fused_vs_oracle(dilqr, port, env, dev, name):
    T, B = (30, 40) if name == "cartpole" else (20, 40)
    pdx, x0, C, c, kw = env_problem(port, name, T, B, torch.float64, sigma=0.05)
    kw["eps"] = 1e-9
    o = port.mpc_forward(x0, port.QuadCost(C, c), pdx, pdx.n_state, pdx.n_ctrl, T, lqr_iter=80,
                         final_pass=False, **kw)
    g = torch.Generator().manual_seed(11)
    gx = torch.randn(o.x.shape, generator=g, dtype=torch.float64)
    gu = torch.randn(o.u.shape, generator=g, dtype=torch.float64)
    ref = port.dilqr_backward(gx, gu, x0, C, c, o.x, o.u, pdx, pdx.n_state, pdx.n_ctrl, pdx.lower,
                              pdx.upper, n_passes=40, tol=1e-15)
    a = _solve_and_grad(dilqr, env, dev, name, T, B, port, True, lqr_iter=80)
    # multi-iteration solves: see test_gpu_parity.test_dilqr_gradient_vs_oracle (1e-8) and
    # test_teacher_forced.py for the per-iteration 1e-10 statement
    assert rel(a[0], o.x) < 1e-8 and rel(a[1], o.u) < 1e-8
    assert rel(a[2], ref.dtheta.sum(0)) < 1e-7
    assert rel(a[3], ref.dC) < 1e-7 and rel(a[4], ref.dc) < 1e-7


@pytest.mark.parametrize("B", [64, 45])
def test_tiled_cost_gradient_reduced_in_kernel(dilqr, env, dev, B):
    """il.tile_cost -> mpc_explicit.MPC -> loss.backward(): (dq, dp) accumulated inside the
    final adjoint pass == the dense dC, dc pushed through TileCost.backward."""
    il = importlib.import_module("differentiable-ilqr_b200.il")
    T = 25
    g = torch.Generator().manual_seed(3)
    r = (torch.rand(B, 4, generator=g, dtype=torch.float64) * 2 - 1) * 0.1
    x0 = torch.stack((r[:, 0], r[:, 1], torch.cos(r[:, 2]), torch.sin(r[:, 2]), r[:, 3]), 1).to(dev)
    uexp = torch.randn(T, B, 1, generator=g, dtype=torch.float64).to(dev)
    proto = env.CartpoleDx()
    q0, p0 = [t.double().to(dev) for t in proto.get_true_obj()]
    out = []
    for tagged in (True, False):
        q, p = q0.clone().requires_grad_(), p0.clone().requires_grad_()
        theta = torch.tensor((9.8, 1.0, 0.1, 0.5), dtype=torch.float64, device=dev, requires_grad=True)
        m = dilqr.mpc_explicit.MPC(5, 1, T, u_lower=proto.lower, u_upper=proto.upper, lqr_iter=60,
                                   verbose=-1, exit_unconverged=False, detach_unconverged=False,
                                   linesearch_decay=proto.linesearch_decay,
                                   max_linesearch_iter=proto.max_linesearch_iter, eps=1e-9,
                                   richardson_passes=30, richardson_tol=None, n_batch=B)
        C, c = il.tile_cost(q, p, T, B) if tagged else il.TileCost.apply(q, p, T, B)
        x, u, _ = m(x0, dilqr.QuadCost(C, c), env.CartpoleDx(theta))
        (u - uexp).pow(2).mean().backward()
        out.append((q.grad.clone(), p.grad.clone(), theta.grad.clone()))
    for a, b in zip(*out):
        assert rel(a, b) < 1e-12, rel(a, b)
    assert float(out[0][0].abs().max()) > 0 and float(out[0][2].abs().max()) > 0


def test_imitation_step_deferred_equals_immediate(dilqr, env, dev):
    """ImitationStep with every validation read deferred to one sync == immediate checks."""
    il = importlib.import_module("differentiable-ilqr_b200.il")
    T, B = 50, 256
    g = torch.Generator().manual_seed(0)
    r = (torch.rand(B, 4, generator=g, dtype=torch.float64) * 2 - 1) * 0.5
    x0 = torch.stack((r[:, 0], r[:, 1], torch.cos(r[:, 2]), torch.sin(r[:, 2]), r[:, 3]), 1)
    uexp = torch.randn(T, B, 1, generator=g, dtype=torch.float64)
    q, p = [t.double() for t in env.CartpoleDx().get_true_obj()]
    theta = torch.tensor((9.8, 1.0, 0.1, 0.5), dtype=torch.float64)
    outs = []
    for defer in (True, False):
        step = il.ImitationStep(env.CartpoleDx, T=T, lqr_iter=10, dtype=torch.float64, device=dev,
                                n_richardson=4)
        step.defer = defer
        outs.append(step.run_host(x0.pin_memory(), uexp.pin_memory(), q.pin_memory(),
                                  p.pin_memory(), theta.pin_memory()))
        assert step.redone == 0
        assert step.mpc.last_info.n_iters == 10
        assert step.mpc.last_backward["fused"]
    assert torch.equal(outs[0], outs[1])
    assert torch.isfinite(outs[0]).all()


def test_expanded_4d_cost_gradient(dilqr, port, env, dev):
    """ADVICE r1: a 4-D stride-0 cost (Q[None,None].expand(T,B,n,n)) through
    mpc_explicit.MPC backward -- the gradient reaches Q summed over (t, b), as the
    reference's autograd does."""
    T, B = 15, 24
    pdx, x0, C, c, kw = env_problem(port, "pendulum", T, B, torch.float64, sigma=0.3)
    kw["eps"] = 1e-9
    outs = []
    for expanded in (True, False):
        Q = C[0, 0].clone().to(dev).requires_grad_()
        pv = c[0, 0].clone().to(dev).requires_grad_()
        if expanded:
            Cc, cc = Q[None, None].expand(T, B, 4, 4), pv[None, None].expand(T, B, 4)
        else:
            Cc, cc = Q[None, None].repeat(T, B, 1, 1), pv[None, None].repeat(T, B, 1)
        theta = pdx.params.to(dev).requires_grad_()
        m = dilqr.mpc_explicit.MPC(3, 1, T, lqr_iter=60, verbose=-1, exit_unconverged=False,
                                   detach_unconverged=False, richardson_passes=40, **kw)
        x, u, _ = m(x0.to(dev), dilqr.QuadCost(Cc, cc), env.PendulumDx(theta))
        (x.sum() + u.pow(2).sum()).backward()
        outs.append((Q.grad.clone(), pv.grad.clone(), theta.grad.clone()))
    for a, b in zip(*outs):
        assert rel(a, b) < 1e-12


def test_host_resident_theta_gets_host_gradient(dilqr, env, dev):
    """ADVICE r1: PendulumDx() keeps its default params on the host with requires_grad;
    the learn_cost flow (il_exp.py:326-336) backpropagates to q, p through
    IL_Env.mpc(env.true_dx, ...) without a device mismatch."""
    il_env = importlib.import_module("differentiable-ilqr_b200.il_env")
    e = il_env.IL_Env("pendulum", lqr_iter=30, mpc_T=10, dtype=torch.float64, device=dev)
    e.true_dx.params.requires_grad_()
    q, p = [t.double().requires_grad_() for t in e.true_dx.get_true_obj()]
    torch.manual_seed(0)
    x0 = e.sample_xinit(6)
    x, u = e.mpc(e.true_dx, x0, q, p)
    u.pow(2).sum().backward()
    assert q.grad is not None and q.grad.device.type == "cpu"
    assert e.true_dx.params.grad is not None and e.true_dx.params.grad.device.type == "cpu"
    assert torch.isfinite(q.grad).all() and torch.isfinite(e.true_dx.params.grad).all()


def test_lqr_step_explicit_entry(dilqr, port, env, dev):
    """lqr_step_explicit.LQRStep(..., no_op_forward=True)(x_init, C, c, F, f, theta): the
    reference's own entry to the DiLQR backward (lqr_step_explicit.py:24-44, 599-712) gives
    the gradients mpc_explicit.MPC gives at the same solution."""
    T, B = 20, 32
    pdx, x0, C, c, kw = env_problem(port, "cartpole", T, B, torch.float64, sigma=0.05)
    kw["eps"] = 1e-9
    g = torch.Generator().manual_seed(4)
    gx = torch.randn(T, B, 5, generator=g, dtype=torch.float64).to(dev)
    gu = torch.randn(T, B, 1, generator=g, dtype=torch.float64).to(dev)
    th1 = pdx.params.to(dev).requires_grad_()
    C1, c1 = C.to(dev).requires_grad_(), c.to(dev).requires_grad_()
    m = dilqr.mpc_explicit.MPC(5, 1, T, lqr_iter=60, verbose=-1, exit_unconverged=False,
                               detach_unconverged=False, richardson_passes=30, **kw)
    x, u, _ = m(x0.to(dev), dilqr.QuadCost(C1, c1), env.CartpoleDx(th1))
    ((x * gx).sum() + (u * gu).sum()).backward()
    th2 = pdx.params.to(dev).requires_grad_()
    C2, c2 = C.to(dev).requires_grad_(), c.to(dev).requires_grad_()
    dx2 = env.CartpoleDx(th2)
    step = dilqr.lqr_step_explicit.LQRStep(
        5, 1, T, u_lower=pdx.lower, u_upper=pdx.upper, true_cost=dilqr.QuadCost(C2, c2),
        true_dynamics=dx2, current_x=x.detach(), current_u=u.detach(), no_op_forward=True)
    F, f = dx2.linearize_traj(x.detach(), u.detach())
    xs, us = step(x0.to(dev), C2, c2, F, f, th2)
    assert torch.equal(xs, x.detach()) and torch.equal(us, u.detach())
    ((xs * gx).sum() + (us * gu).sum()).backward()
    assert rel(th2.grad, th1.grad) < 1e-10
    assert rel(C2.grad, C1.grad) < 1e-10 and rel(c2.grad, c1.grad) < 1e-10
    # and one real step (lqr_step_explicit.py:620-650) == lqr_step.LQRStep on the same iterate
    u0 = torch.zeros(T, B, 1, dtype=torch.float64, device=dev)
    x_roll = dilqr.util.get_traj(T, u0, x0.to(dev), env.CartpoleDx(pdx.params.to(dev)))
    a = dilqr.lqr_step_explicit.LQRStep(5, 1, T, u_lower=pdx.lower, u_upper=pdx.upper,
                                        true_dynamics=env.CartpoleDx(pdx.params.to(dev)),
                                        current_x=x_roll, current_u=u0,
                                        linesearch_decay=pdx.linesearch_decay,
                                        max_linesearch_iter=pdx.max_linesearch_iter)(
        x0.to(dev), C.to(dev), c.to(dev))
    b = dilqr.LQRStep(5, 1, T, u_lower=pdx.lower, u_upper=pdx.upper,
                      true_dynamics=env.CartpoleDx(pdx.params.to(dev)), current_x=x_roll,
                      current_u=u0, linesearch_decay=pdx.linesearch_decay,
                      max_linesearch_iter=pdx.max_linesearch_iter)(
        x0.to(dev), C.to(dev), c.to(dev), None)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])

