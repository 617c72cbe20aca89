#!/usr/bin/env python
"""Generate the golden vectors in tests/golden/*.npz by running the UNMODIFIED
reference (/root/reference, imported through oracle/ref_harness.py).

Build-container only (the reference does not travel to the GPU box); the
resulting small .npz files are committed and are what the tests read.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py
"""
import os
import pickle
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_harness  # noqa: E402
sys.path.insert(0, os.path.join(ROOT, "tests"))
from common import SoftCost as _SoftCost, SoftDyn as _SoftDyn  # noqa: E402

R = ref_harness.load()


def npz(name, **kw):
    out = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v))
           for k, v in kw.items()}
    np.savez_compressed(os.path.join(HERE, name), **out)
    print("wrote", name, {k: v.shape for k, v in out.items()})


def fixtures():
    """The reference's own data/*.pkl expert trajectories (SURVEY 8c)."""
    for env in ("cartpole", "pendulum"):
        e = pickle.load(open(os.path.join(ref_harness.REF_ROOT, "data", env + ".pkl"), "rb"))
        tau = torch.cat((e.train_data, e.val_data, e.test_data), 0).detach()
        npz("fixture_%s.npz" % env, tau=tau, mpc_T=e.mpc_T, lqr_iter=e.lqr_iter)


def lindx(boxed):
    torch.manual_seed(0)
    torch.set_default_dtype(torch.float64)
    ns, nc, T, B = 4, 2, 12, 16
    n = ns + nc
    A = torch.randn(T, B, n, n)
    C = A.transpose(2, 3) @ A + torch.eye(n)
    c = torch.randn(T, B, n)
    F = torch.cat((torch.eye(ns).expand(T - 1, B, ns, ns) + 0.2 * torch.randn(T - 1, B, ns, ns) / ns ** 0.5,
                   torch.randn(T - 1, B, ns, nc) / ns ** 0.5), 3)
    f = 0.1 * torch.randn(T - 1, B, ns)
    x0 = torch.randn(B, ns)
    kw = dict(u_lower=-1.0, u_upper=1.0) if boxed else {}
    Cg, cg, Fg, fg, x0g = [t.clone().requires_grad_() for t in (C, c, F, f, x0)]
    m = R.mpc.MPC(ns, nc, T, lqr_iter=20, verbose=-1, exit_unconverged=False, **kw)
    x, u, costs = m(x0g, R.mpc.QuadCost(Cg, cg), R.mpc.LinDx(Fg, fg))
    g = torch.Generator().manual_seed(7)
    gx = torch.randn(x.shape, generator=g)
    gu = torch.randn(u.shape, generator=g)
    ((x * gx).sum() + (u * gu).sum()).backward()
    npz("ref_lindx_%s.npz" % ("boxed" if boxed else "free"), C=C, c=c, F=F, f=f, x0=x0, x=x, u=u,
        costs=costs, gx=gx, gu=gu, dx0=x0g.grad, dC=Cg.grad, dc=cg.grad, dF=Fg.grad, df=fg.grad)


def slew_affine():
    """mpc.MPC with slew_rate_penalty + prev_ctrl on a LinDx problem (mpc.py:362-445) and
    with dynamics.AffineDynamics (dynamics.py:159-202), forward and KKT gradients."""
    torch.manual_seed(11)
    torch.set_default_dtype(torch.float64)
    ns, nc, T, B = 4, 2, 10, 6
    n = ns + nc
    A = torch.randn(T, B, n, n)
    C = A.transpose(2, 3) @ A + torch.eye(n)
    c = torch.randn(T, B, n)
    F = torch.cat((torch.eye(ns).expand(T - 1, B, ns, ns) + 0.2 * torch.randn(T - 1, B, ns, ns) / ns ** 0.5,
                   torch.randn(T - 1, B, ns, nc) / ns ** 0.5), 3)
    f = 0.1 * torch.randn(T - 1, B, ns)
    x0 = torch.randn(B, ns)
    prev = 0.3 * torch.randn(B, nc)
    g = torch.Generator().manual_seed(7)
    gx = torch.randn(T, B, ns, generator=g)
    gu = torch.randn(T, B, nc, generator=g)
    out = dict(C=C, c=c, F=F, f=f, x0=x0, prev=prev, gx=gx, gu=gu)
    # affine dynamics, time-invariant
    import dynamics as refdyn
    Am = (torch.eye(ns) + 0.2 * torch.randn(ns, ns) / ns ** 0.5).requires_grad_()
    Bm = (torch.randn(ns, nc) / ns ** 0.5).requires_grad_()
    cm = (0.1 * torch.randn(ns)).requires_grad_()
    Cg, cg, x0g = [t.clone().requires_grad_() for t in (C, c, x0)]
    m = R.mpc.MPC(ns, nc, T, lqr_iter=20, verbose=-1, exit_unconverged=False, u_lower=-1.0,
                  u_upper=1.0, grad_method=R.mpc.GradMethods.ANALYTIC)
    x, u, costs = m(x0g, R.mpc.QuadCost(Cg, cg), refdyn.AffineDynamics(Am, Bm, cm))
    ((x * gx).sum() + (u * gu).sum()).backward()
    out.update(A=Am, B=Bm, cvec=cm, a_x=x, a_u=u, a_costs=costs, a_dx0=x0g.grad, a_dC=Cg.grad,
               a_dc=cg.grad, a_dA=Am.grad, a_dB=Bm.grad, a_dcvec=cm.grad)
    # slew-rate penalty: the reference's LinDx branch is broken (true_dynamics=None is called,
    # lqr_step.py:224), the Module-dynamics branch (CtrlPassthroughDynamics) works
    Am2, Bm2, cm2 = [t.detach().clone().requires_grad_() for t in (Am, Bm, cm)]
    Cg, cg, x0g = [t.clone().requires_grad_() for t in (C, c, x0)]
    m = R.mpc.MPC(ns, nc, T, lqr_iter=20, verbose=-1, exit_unconverged=False, u_lower=-1.0,
                  u_upper=1.0, slew_rate_penalty=0.4, prev_ctrl=prev,
                  grad_method=R.mpc.GradMethods.ANALYTIC)
    x, u, costs = m(x0g, R.mpc.QuadCost(Cg, cg), refdyn.AffineDynamics(Am2, Bm2, cm2))
    ((x * gx).sum() + (u * gu).sum()).backward()
    out.update(s_x=x, s_u=u, s_costs=costs, s_dx0=x0g.grad, s_dC=Cg.grad, s_dc=cg.grad,
               s_dA=Am2.grad, s_dB=Bm2.grad, s_dcvec=cm2.grad)
    npz("ref_slew_affine.npz", **out)
    torch.set_default_dtype(torch.float32)


def dilqr(env, T, B, lqr_iter, sigma):
    torch.manual_seed(0)
    torch.set_default_dtype(torch.float64)
    dt = torch.float64
    if env == "pendulum":
        theta = torch.tensor((10., 1., 1.), dtype=dt, requires_grad=True)
        dx = R.pendulum.PendulumDx(theta)
        th = (torch.rand(B) - 0.5) * 3.14159
        w = torch.rand(B) * 2 - 1
        x0 = torch.stack((torch.cos(th), torch.sin(th), w), 1)
    elif env == "rocket":
        theta = torch.tensor((0.5, 1.0, 1.0, 1.0, 1.0), dtype=dt, requires_grad=True)
        dx = R.rocket.RocketDx(theta)
        dx.lower, dx.upper = -20.0, 20.0          # float bounds (SURVEY 8d config 3)
        qv = torch.cat((torch.ones(B, 1), 0.1 * torch.randn(B, 3)), 1)
        x0 = torch.cat(((torch.rand(B, 3) * 2 - 1) * 3, torch.rand(B, 3) * 2 - 1,
                        qv / qv.norm(dim=1, keepdim=True), (torch.rand(B, 3) * 2 - 1) * 0.1), 1)
    else:
        theta = torch.tensor((9.8, 1.0, 0.1, 0.5), dtype=dt, requires_grad=True)
        dx = R.cartpole.CartpoleDx(theta)
        r = (torch.rand(B, 4) * 2 - 1) * sigma
        x0 = torch.stack((r[:, 0], r[:, 1], torch.cos(r[:, 2]), torch.sin(r[:, 2]), r[:, 3]), 1)
    q, p = dx.get_true_obj()
    q, p = q.to(dt), p.to(dt)
    C = torch.diag(q)[None, None].repeat(T, B, 1, 1).requires_grad_()
    c = p[None, None].repeat(T, B, 1).requires_grad_()
    m = R.mpc_explicit.MPC(dx.n_state, dx.n_ctrl, T, u_lower=dx.lower, u_upper=dx.upper,
                           lqr_iter=lqr_iter, verbose=-1, exit_unconverged=False,
                           detach_unconverged=False, linesearch_decay=dx.linesearch_decay,
                           max_linesearch_iter=dx.max_linesearch_iter, eps=1e-9,
                           grad_method=R.mpc_explicit.GradMethods.ANALYTIC)
    x, u, costs = m(x0, R.mpc_explicit.QuadCost(C, c), dx)
    g = torch.Generator().manual_seed(7)
    gx = torch.randn(x.shape, generator=g)
    gu = torch.randn(u.shape, generator=g)
    ((x * gx).sum() + (u * gu).sum()).backward()
    npz("ref_dilqr_%s.npz" % env, x0=x0, q=q, p=p, theta=theta.detach(), x=x, u=u, costs=costs,
        gx=gx, gu=gu, dC=C.grad, dc=c.grad, dtheta=theta.grad, T=T, lqr_iter=lqr_iter)


def dilqr_t50(B=16, sigma=0.05, presolve=250):
    """DiLQR gradient at the HEADLINE horizon (cartpole T=50) in the regime where the
    implicit gradient is well posed (SURVEY 8d config 2b): perturbation +-0.05, controls
    warm-started from an untimed pre-solve, so the differentiated solve stops after one
    iteration at a converged fixed point.  T*B = 800 < 1000 keeps the reference on its CPU
    KKT_gradient path (lqr_step_explicit.py:664-705)."""
    torch.manual_seed(0)
    torch.set_default_dtype(torch.float64)
    dt = torch.float64
    T = 50
    theta = torch.tensor((9.8, 1.0, 0.1, 0.5), dtype=dt, requires_grad=True)
    dx = R.cartpole.CartpoleDx(theta)
    r = (torch.rand(B, 4) * 2 - 1) * sigma
    x0 = torch.stack((r[:, 0], r[:, 1], torch.cos(r[:, 2]), torch.sin(r[:, 2]), r[:, 3]), 1)
    q, p = dx.get_true_obj()
    q, p = q.to(dt), p.to(dt)
    kw = dict(u_lower=dx.lower, u_upper=dx.upper, verbose=-1, exit_unconverged=False,
              detach_unconverged=False, linesearch_decay=dx.linesearch_decay,
              max_linesearch_iter=dx.max_linesearch_iter, eps=1e-9,
              grad_method=R.mpc_explicit.GradMethods.ANALYTIC)
    C0 = torch.diag(q)[None, None].repeat(T, B, 1, 1)
    c0 = p[None, None].repeat(T, B, 1)
    with torch.no_grad():
        pre = R.mpc_explicit.MPC(dx.n_state, dx.n_ctrl, T, lqr_iter=presolve, **kw)
        _, u_warm, _ = pre(x0, R.mpc_explicit.QuadCost(C0, c0), R.cartpole.CartpoleDx(theta.detach()))
    C = C0.clone().requires_grad_()
    c = c0.clone().requires_grad_()
    m = R.mpc_explicit.MPC(dx.n_state, dx.n_ctrl, T, lqr_iter=5, u_init=u_warm.clone(), **kw)
    x, u, costs = m(x0, R.mpc_explicit.QuadCost(C, c), dx)
    g = torch.Generator().manual_seed(7)
    gx = torch.randn(x.shape, generator=g)
    gu = torch.randn(u.shape, generator=g)
    ((x * gx).sum() + (u * gu).sum()).backward()
    npz("ref_dilqr_cartpole_T50.npz", x0=x0, q=q, p=p, theta=theta.detach(), u_init=u_warm, x=x,
        u=u, costs=costs, gx=gx, gu=gu, dC=C.grad, dc=c.grad, dtheta=theta.grad, T=T, lqr_iter=5,
        du_warm=(u - u_warm).abs().max())
    torch.set_default_dtype(torch.float32)


def module_cost_and_dynamics():
    """mpc.MPC with a cost Module (approximate_cost, mpc.py:447-487) on LinDx dynamics, and with
    a dynamics Module under AUTO_DIFF / FINITE_DIFF (mpc.py:525-601) on a QuadCost: forward
    solutions and the gradients wrt the Modules' parameters."""
    torch.set_default_dtype(torch.float64)
    out = {}
    ns, nc, T, B = 4, 2, 8, 6
    n = ns + nc
    g = torch.Generator().manual_seed(21)
    F = (torch.eye(ns).unsqueeze(0).unsqueeze(0).repeat(T - 1, B, 1, 1)
         + 0.2 * torch.randn(T - 1, B, ns, ns, generator=g))
    F = torch.cat((F, torch.randn(T - 1, B, ns, nc, generator=g)), 3)
    f = 0.1 * torch.randn(T - 1, B, ns, generator=g)
    x0 = torch.randn(B, ns, generator=g)
    gx = torch.randn(T, B, ns, generator=g)
    gu = torch.randn(T, B, nc, generator=g)
    cost = _SoftCost(n, 5)
    Fg, fg, x0g = F.clone().requires_grad_(), f.clone().requires_grad_(), x0.clone().requires_grad_()
    m = R.mpc.MPC(ns, nc, T, u_lower=-1.0, u_upper=1.0, lqr_iter=20, verbose=-1, n_batch=B,
                  exit_unconverged=False, detach_unconverged=False, eps=1e-9, backprop=True,
                  max_linesearch_iter=10, linesearch_decay=0.2)
    x, u, costs = m(x0g, cost, R.mpc.LinDx(Fg, fg))
    ((x * gx).sum() + (u * gu).sum()).backward()
    out.update(c_F=F, c_f=f, c_x0=x0, c_gx=gx, c_gu=gu, c_x=x, c_u=u, c_costs=costs,
               c_dA=cost.A.grad, c_dp=cost.p.grad, c_dw=cost.w.grad, c_dF=Fg.grad, c_df=fg.grad,
               c_dx0=x0g.grad)
    # dynamics Module, two linearisation methods
    q = torch.cat((torch.ones(ns), 0.1 * torch.ones(nc)))
    Cq = torch.diag(q)[None, None].repeat(T, B, 1, 1)
    cq = 0.3 * torch.randn(T, B, n, generator=g)
    for name, gm in (("ad", R.mpc.GradMethods.AUTO_DIFF), ("fd", R.mpc.GradMethods.FINITE_DIFF)):
        dyn = _SoftDyn(ns, nc, 9)
        Cg, cg = Cq.clone().requires_grad_(), cq.clone().requires_grad_()
        m = R.mpc.MPC(ns, nc, T, u_lower=-1.0, u_upper=1.0, lqr_iter=20, verbose=-1, n_batch=B,
                      exit_unconverged=False, detach_unconverged=False, eps=1e-9, grad_method=gm,
                      max_linesearch_iter=10, linesearch_decay=0.2)
        x, u, costs = m(x0, R.mpc.QuadCost(Cg, cg), dyn)
        ((x * gx).sum() + (u * gu).sum()).backward()
        out.update({"d_%s_x" % name: x, "d_%s_u" % name: u, "d_%s_costs" % name: costs,
                    "d_%s_dA" % name: dyn.A.grad, "d_%s_dB" % name: dyn.B.grad,
                    "d_%s_dW" % name: dyn.W.grad, "d_%s_dC" % name: Cg.grad, "d_%s_dc" % name: cg.grad})
    out.update(d_C=Cq, d_c=cq)
    npz("ref_module_cost_dynamics.npz", **out)
    torch.set_default_dtype(torch.float32)


def tables():
    torch.manual_seed(1)
    torch.set_default_dtype(torch.float64)
    out = {}
    for env, cls, ns, nth in (("cartpole", R.cartpole.CartpoleDx, 5, 4),
                              ("pendulum", R.pendulum.PendulumDx, 3, 3),
                              ("rocket", R.rocket.RocketDx, 13, 5)):
        theta = torch.rand(nth) * 2 + 0.3
        dx = cls(theta.clone())
        x = torch.randn(6, ns)
        u = torch.randn(6, dx.n_ctrl)
        names = ["D", "D_theta", "D_x", "D_u", "x_theta", "x_x", "x_u"]
        res = dx.get_matrices(x, u)
        out.update({env + "_theta": theta, env + "_x": x, env + "_u": u})
        out.update({env + "_" + n: t for n, t in zip(names, res)})
        out[env + "_step"] = dx(x, u)
        out[env + "_lin"] = dx.get_linear_dyn(x, u)
    npz("ref_tables.npz", **out)


def env_forward(env, T, B, lqr_iter, dtype):
    """Forward-only env solve incl. per-iteration qp counts (control-flow parity)."""
    torch.manual_seed(3)
    torch.set_default_dtype(dtype)
    if env == "pendulum":
        dx = R.pendulum.PendulumDx(torch.tensor((10., 1., 1.), dtype=dtype))
        th = (torch.rand(B) - 0.5) * 3.14159
        w = torch.rand(B) * 2 - 1
        x0 = torch.stack((torch.cos(th), torch.sin(th), w), 1)
    else:
        dx = R.cartpole.CartpoleDx(torch.tensor((9.8, 1.0, 0.1, 0.5), dtype=dtype))
        r = (torch.rand(B, 4) * 2 - 1) * 0.5
        x0 = torch.stack((r[:, 0], r[:, 1], torch.cos(r[:, 2]), torch.sin(r[:, 2]), r[:, 3]), 1)
    q, p = dx.get_true_obj()
    C = torch.diag(q.to(dtype))[None, None].repeat(T, B, 1, 1)
    c = p.to(dtype)[None, None].repeat(T, B, 1)
    m = R.mpc_explicit.MPC(dx.n_state, dx.n_ctrl, T, u_lower=dx.lower, u_upper=dx.upper,
                           lqr_iter=lqr_iter, verbose=-1, exit_unconverged=False,
                           detach_unconverged=False, linesearch_decay=dx.linesearch_decay,
                           max_linesearch_iter=dx.max_linesearch_iter, eps=dx.mpc_eps,
                           grad_method=R.mpc_explicit.GradMethods.ANALYTIC)
    with torch.no_grad():
        try:
            x, u, costs = m(x0, R.mpc_explicit.QuadCost(C, c), dx)
        except RuntimeError:
            raise
    tag = "f64" if dtype == torch.float64 else "f32"
    npz("ref_fwd_%s_%s.npz" % (env, tag), x0=x0, q=q.to(dtype), p=p.to(dtype), x=x, u=u,
        costs=costs, T=T, lqr_iter=lqr_iter)
    torch.set_default_dtype(torch.float32)


def nn_dynamics():
    """mpc.MPC with dynamics.NNDynamics (one hidden layer, ANALYTIC linearisation): forward
    and the KKT gradients wrt the network weights, the cost and x_init."""
    import dynamics as refdyn
    torch.set_default_dtype(torch.float64)
    out = {}
    for act in ("sigmoid", "relu"):
        torch.manual_seed(5)
        ns, nc, T, B = 3, 1, 10, 7
        n = ns + nc
        dx = refdyn.NNDynamics(ns, nc, hidden_sizes=[12], activation=act, passthrough=True)
        for p_ in dx.parameters():
            p_.data.mul_(0.5)
        A = torch.randn(T, B, n, n)
        C = A.transpose(2, 3) @ A + torch.eye(n)
        c = torch.randn(T, B, n)
        x0 = torch.randn(B, ns)
        g = torch.Generator().manual_seed(7)
        gx = torch.randn(T, B, ns, generator=g)
        gu = torch.randn(T, B, nc, generator=g)
        Cg, cg, x0g = [t.clone().requires_grad_() for t in (C, c, x0)]
        m = R.mpc.MPC(ns, nc, T, lqr_iter=30, verbose=-1, exit_unconverged=False, u_lower=-1.0,
                      u_upper=1.0, grad_method=R.mpc.GradMethods.ANALYTIC, detach_unconverged=False)
        x, u, costs = m(x0g, R.mpc.QuadCost(Cg, cg), dx)
        ((x * gx).sum() + (u * gu).sum()).backward()
        W1, b1, W2, b2 = dx.fcs[0].weight, dx.fcs[0].bias, dx.fcs[1].weight, dx.fcs[1].bias
        out.update({act + "_" + k: v for k, v in dict(
            C=C, c=c, x0=x0, gx=gx, gu=gu, W1=W1, b1=b1, W2=W2, b2=b2, x=x, u=u, costs=costs,
            dC=Cg.grad, dc=cg.grad, dx0=x0g.grad, dW1=W1.grad, db1=b1.grad, dW2=W2.grad,
            db2=b2.grad).items()})
    npz("ref_nn_dynamics.npz", **out)
    torch.set_default_dtype(torch.float32)


def nn_two_layers():
    """mpc.MPC + NNDynamics(hidden_sizes=[10, 6]) (dynamics.py:98-116, two factors in
    grad_input), forward and KKT gradients wrt all six parameter tensors."""
    import dynamics as refdyn
    torch.set_default_dtype(torch.float64)
    out = {}
    for act in ("sigmoid", "relu"):
        torch.manual_seed(21)
        ns, nc, T, B = 3, 1, 8, 5
        n = ns + nc
        dx = refdyn.NNDynamics(ns, nc, hidden_sizes=[10, 6], activation=act, passthrough=True)
        for p_ in dx.parameters():
            p_.data.mul_(0.5)
        A = torch.randn(T, B, n, n)
        C = A.transpose(2, 3) @ A + torch.eye(n)
        c = torch.randn(T, B, n)
        x0 = torch.randn(B, ns)
        g = torch.Generator().manual_seed(7)
        gx = torch.randn(T, B, ns, generator=g)
        gu = torch.randn(T, B, nc, generator=g)
        for L in (1, 40):
            Cg = C.clone().requires_grad_()
            for p_ in dx.parameters():
                p_.grad = None
            m = R.mpc.MPC(ns, nc, T, lqr_iter=L, verbose=-1, exit_unconverged=(L > 1 and act == "sigmoid"),
                          u_lower=-2.0, u_upper=2.0, grad_method=R.mpc.GradMethods.ANALYTIC,
                          detach_unconverged=(L > 1 and act == "sigmoid"))
            x, u, costs = m(x0, R.mpc.QuadCost(Cg, c), dx)
            out.update({"%s_L%d_%s" % (act, L, k): v for k, v in dict(x=x, u=u, costs=costs).items()})
        ((x * gx).sum() + (u * gu).sum()).backward()
        prm = {"W%d" % (i + 1): fc.weight for i, fc in enumerate(dx.fcs)}
        prm.update({"b%d" % (i + 1): fc.bias for i, fc in enumerate(dx.fcs)})
        out.update({act + "_" + k: v for k, v in dict(C=C, c=c, x0=x0, gx=gx, gu=gu, dC=Cg.grad).items()})
        out.update({act + "_" + k: v for k, v in prm.items()})
        out.update({act + "_d" + k: v.grad for k, v in prm.items()})
    npz("ref_nn_two_layers.npz", **out)
    torch.set_default_dtype(torch.float32)


def nn_grad_methods():
    """mpc.MPC + NNDynamics with grad_method AUTO_DIFF and FINITE_DIFF (mpc.py:525-601)."""
    import dynamics as refdyn
    torch.set_default_dtype(torch.float64)
    out = {}
    for name, gm in (("auto", R.mpc.GradMethods.AUTO_DIFF), ("fd", R.mpc.GradMethods.FINITE_DIFF)):
        torch.manual_seed(9)
        ns, nc, T, B = 3, 1, 6, 4
        n = ns + nc
        dx = refdyn.NNDynamics(ns, nc, hidden_sizes=[8], activation="sigmoid", passthrough=True)
        for p_ in dx.parameters():
            p_.data.mul_(0.5)
        A = torch.randn(T, B, n, n)
        C = A.transpose(2, 3) @ A + torch.eye(n)
        c = torch.randn(T, B, n)
        x0 = torch.randn(B, ns)
        g = torch.Generator().manual_seed(7)
        gx = torch.randn(T, B, ns, generator=g)
        gu = torch.randn(T, B, nc, generator=g)
        Cg = C.clone().requires_grad_()
        # exit_unconverged=True + detach_unconverged=True: the reference asserts that every
        # problem reached max|du| < eps, so the golden is a converged solve
        m = R.mpc.MPC(ns, nc, T, lqr_iter=40, verbose=-1, exit_unconverged=True, u_lower=-2.0,
                      u_upper=2.0, grad_method=gm, detach_unconverged=True)
        x, u, costs = m(x0, R.mpc.QuadCost(Cg, c), dx)
        ((x * gx).sum() + (u * gu).sum()).backward()
        W1, b1, W2, b2 = dx.fcs[0].weight, dx.fcs[0].bias, dx.fcs[1].weight, dx.fcs[1].bias
        out.update({name + "_" + k: v for k, v in dict(
            C=C, c=c, x0=x0, gx=gx, gu=gu, W1=W1, b1=b1, W2=W2, b2=b2, x=x, u=u, costs=costs,
            dC=Cg.grad, dW1=W1.grad, db1=b1.grad, dW2=W2.grad, db2=b2.grad).items()})
    npz("ref_nn_grad_methods.npz", **out)
    torch.set_default_dtype(torch.float32)


def delta_u():
    """mpc.MPC with the delta_u trust region (lqr_step.py:132-134,204-211) on a boxed LinDx
    problem: forward + KKT gradients."""
    torch.manual_seed(13)
    torch.set_default_dtype(torch.float64)
    ns, nc, T, B = 4, 2, 10, 8
    n = ns + nc
    A = torch.randn(T, B, n, n)
    C = A.transpose(2, 3) @ A + torch.eye(n)
    c = torch.randn(T, B, n)
    F = torch.cat((torch.eye(ns).expand(T - 1, B, ns, ns) + 0.2 * torch.randn(T - 1, B, ns, ns) / ns ** 0.5,
                   torch.randn(T - 1, B, ns, nc) / ns ** 0.5), 3)
    f = 0.1 * torch.randn(T - 1, B, ns)
    x0 = torch.randn(B, ns)
    g = torch.Generator().manual_seed(7)
    gx = torch.randn(T, B, ns, generator=g)
    gu = torch.randn(T, B, nc, generator=g)
    out = dict(C=C, c=c, F=F, f=f, x0=x0, gx=gx, gu=gu)
    for L in (1, 3, 25):
        Cg, cg, Fg, fg, x0g = [t.clone().requires_grad_() for t in (C, c, F, f, x0)]
        m = R.mpc.MPC(ns, nc, T, lqr_iter=L, verbose=-1, exit_unconverged=False, u_lower=-1.0,
                      u_upper=1.0, delta_u=0.25, detach_unconverged=False)
        x, u, costs = m(x0g, R.mpc.QuadCost(Cg, cg), R.mpc.LinDx(Fg, fg))
        out.update({"L%d_x" % L: x, "L%d_u" % L: u, "L%d_costs" % L: costs})
        if L == 25:
            ((x * gx).sum() + (u * gu).sum()).backward()
            out.update(dx0=x0g.grad, dC=Cg.grad, dc=cg.grad, dF=Fg.grad, df=fg.grad)
    npz("ref_delta_u.npz", **out)
    torch.set_default_dtype(torch.float32)


PNQP_CASES = ((1, 0), (2, 1), (3, 2), (4, 3))      # (n, seed)


def pnqp_cases():
    """pnqp.pnqp (pnqp.py) on random box-constrained QPs, B=32, cold and warm started.

    The committed ref_pnqp.npz was written by this function with oracle/port.py's pnqp in
    place of the reference's (the reference tree was no longer at hand); on exactly these
    cases the two had been compared directly and agreed bit for bit (x, If, iteration
    count).  Rerunning this function regenerates the file from the reference itself."""
    torch.set_default_dtype(torch.float64)
    out = {}
    for n, seed in PNQP_CASES:
        torch.manual_seed(seed)
        B = 32
        A = torch.randn(B, n, n)
        H = A.transpose(1, 2) @ A + 0.5 * torch.eye(n)
        q = 2 * torch.randn(B, n)
        lo, hi = -torch.rand(B, n), torch.rand(B, n)
        k = "n%d_s%d_" % (n, seed)
        x_warm = torch.randn(B, n)
        out.update({k + "H": H, k + "q": q, k + "lo": lo, k + "hi": hi, k + "x_init": x_warm})
        for tag, x_init in (("cold", None), ("warm", x_warm)):
            x, _, If, i = R.pnqp.pnqp(H, q, lo, hi, x_init=x_init, n_iter=20)
            out.update({k + tag + "_x": x, k + tag + "_If": If, k + tag + "_n_iter": i})
    npz("ref_pnqp.npz", **out)
    torch.set_default_dtype(torch.float32)


def backup_chol():
    """mpc_backup.MPC (lqr_step_backup: Cholesky(+1e-6 I) gains, used inside the DiLQR
    backward), one iteration on a LinDx problem.

    The committed ref_backup_chol.npz was written by this function with oracle/port.py
    (gain_solve="chol_reg") in place of the reference, which it had matched on exactly this
    case to 1e-13; rerunning this function regenerates the file from the reference."""
    torch.manual_seed(0)
    torch.set_default_dtype(torch.float64)
    ns, nc, T, B = 4, 2, 8, 6
    n = ns + nc
    A = torch.randn(T, B, n, n)
    C = A.transpose(2, 3) @ A + torch.eye(n)
    c = torch.randn(T, B, n)
    F = torch.randn(T - 1, B, ns, n) / 2
    x0 = torch.randn(B, ns)
    m = R.mpc_backup.MPC(ns, nc, T, lqr_iter=1, verbose=-1, exit_unconverged=False)
    x, u, _ = m(x0, R.mpc_backup.QuadCost(C, c), R.mpc_backup.LinDx(F, None))
    npz("ref_backup_chol.npz", C=C, c=c, F=F, x0=x0, x=x, u=u)
    torch.set_default_dtype(torch.float32)


def open_loop(env, mpc_T, lqr_iter, n_train, n_val, n_test):
    """IL_Env.populate_data (il_env.py:81-94): one batched open-loop expert solve."""
    torch.set_default_dtype(torch.float64)
    e = R.il_env.IL_Env(env, lqr_iter=lqr_iter, mpc_T=mpc_T)
    torch.manual_seed(0)
    x0 = e.sample_xinit(n_batch=n_train + n_val + n_test)
    e.populate_data(n_train, n_val, n_test, seed=0)
    npz("ref_open_loop_%s.npz" % env, x0=x0, train=e.train_data, val=e.val_data,
        test=e.test_data, mpc_T=mpc_T, lqr_iter=lqr_iter)
    torch.set_default_dtype(torch.float32)


def closed_loop(env, mpc_T, lqr_iter, n_train, n_val, n_test):
    """IL_Env.populate_data2 (il_env.py:96-151): closed-loop receding-horizon expert data,
    one B=1 MPC call per (sample, step)."""
    torch.set_default_dtype(torch.float64)
    e = R.il_env.IL_Env(env, lqr_iter=lqr_iter, mpc_T=mpc_T)
    torch.manual_seed(0)
    x0 = e.sample_xinit(n_batch=n_train + n_val + n_test)
    e.populate_data2(n_train, n_val, n_test, seed=0)
    npz("ref_closed_loop_%s.npz" % env, x0=x0, train=e.train_data, val=e.val_data,
        test=e.test_data, mpc_T=mpc_T, lqr_iter=lqr_iter)
    torch.set_default_dtype(torch.float32)


if __name__ == "__main__":
    if sys.argv[1:] == ["t50"]:      # only the headline-horizon DiLQR golden (about a minute)
        dilqr_t50()
        sys.exit(0)
    if sys.argv[1:] == ["modules"]:
        module_cost_and_dynamics()
        sys.exit(0)
    fixtures()
    lindx(False)
    lindx(True)
    dilqr("pendulum", 20, 4, 60, None)
    dilqr("cartpole", 12, 8, 80, 0.05)
    dilqr("rocket", 10, 4, 60, None)
    dilqr_t50()
    tables()
    env_forward("cartpole", 25, 16, 6, torch.float64)
    env_forward("pendulum", 20, 16, 8, torch.float64)
    env_forward("cartpole", 25, 16, 6, torch.float32)
    closed_loop("pendulum", 20, 50, 4, 1, 1)
    closed_loop("cartpole", 12, 30, 1, 1, 1)
    slew_affine()
    open_loop("pendulum", 20, 60, 5, 2, 1)
    nn_dynamics()
    nn_grad_methods()
    delta_u()
    nn_two_layers()
    module_cost_and_dynamics()
    pnqp_cases()
    backup_chol()
