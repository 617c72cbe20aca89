"""CPU oracle for the batched differentiable iLQR / MPC hot path.

TEST INFRASTRUCTURE ONLY.  This file is a from-scratch restatement (torch CPU
tensor arithmetic, batch-vectorised exactly like the reference so the
batch-global control flow is reproduced) of the algorithm implemented by the
reference repo josef-w/Differentiable-iLQR.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl
reference`` legs may import it; the product (``differentiable-ilqr_b200``)
never does and has no CPU fallback.

Parity status: PINNED.  ``tests/test_oracle_golden.py`` and
``tests/test_oracle_vs_reference.py`` check this port against the golden
vectors in ``tests/golden`` (generated from the reference by
``tests/golden/make_golden.py``, which imports it through
``oracle/ref_harness.py``; the two ``data/*.pkl`` expert-trajectory fixtures
of the reference are included there).

Every function cites the reference file:line it restates (paths relative to
the reference root).
"""
from collections import namedtuple
import math

import torch

QuadCost = namedtuple("QuadCost", "C c")      # definitions.py:3
LinDx = namedtuple("LinDx", "F f")            # definitions.py:4


# --------------------------------------------------------------------------
# tiny batched helpers (util.py:42-72)
# --------------------------------------------------------------------------
def _mv(M, v):                       # util.py:46  bmv
    return torch.bmm(M, v.unsqueeze(2)).squeeze(2)


def _outer(a, b):                    # util.py:42  bger
    return a.unsqueeze(2) * b.unsqueeze(1)


def _quad(x, Q):                     # util.py:50  bquad
    return torch.bmm(torch.bmm(x.unsqueeze(1), Q), x.unsqueeze(2)).reshape(-1)


def _dot(a, b):                      # util.py:54  bdot
    return torch.bmm(a.unsqueeze(1), b.unsqueeze(2)).reshape(-1)


def _clamp(x, lo, hi):               # util.py:58-72 eclamp (out of place here)
    x = x.clone()
    lo_t = lo if torch.is_tensor(lo) else torch.full_like(x, float(lo))
    hi_t = hi if torch.is_tensor(hi) else torch.full_like(x, float(hi))
    m = x < lo_t
    x[m] = lo_t[m]
    m = x > hi_t
    x[m] = hi_t[m]
    return x


def _bound(v, t):                    # lqr_step.py:264-272 get_bound
    return v if isinstance(v, float) else v[t]


# --------------------------------------------------------------------------
# projected-Newton box QP  (pnqp.py:5-82)
# --------------------------------------------------------------------------
PnqpOut = namedtuple("PnqpOut", "x Hfree If n_iter converged")


def pnqp(H, q, lower, upper, x_init=None, n_iter=20):
    """min 1/2 x'Hx + q'x  s.t. lower <= x <= upper, batched, with the
    reference's *batch-global* termination and Armijo logic (pnqp.py:56-76).
    Returns the masked Hessian ``H_`` (not its LU) as ``Hfree``."""
    GAMMA = 0.1
    B, n, _ = H.shape
    eye = 1e-11 * torch.eye(n, dtype=H.dtype).expand(B, n, n)

    def obj(x):                                        # pnqp.py:11-12
        return 0.5 * _quad(x, H) + _dot(q, x)

    if x_init is None:                                 # pnqp.py:14-19
        if n == 1:
            x0 = -(1.0 / H.squeeze(2)) * q
        else:
            x0 = -torch.linalg.solve(H, q.unsqueeze(2)).squeeze(2)
    else:
        x0 = x_init.clone()
    x = _clamp(x0, lower, upper)                       # pnqp.py:23
    lo_t = lower if torch.is_tensor(lower) else torch.full_like(x, float(lower))
    hi_t = upper if torch.is_tensor(upper) else torch.full_like(x, float(upper))

    H_ = If = None
    for i in range(n_iter):
        g = _mv(H, x) + q                              # pnqp.py:29
        Ic = (((x == lo_t) & (g > 0)) | ((x == hi_t) & (g < 0))).to(H.dtype)
        If = 1 - Ic                                    # pnqp.py:32-33
        Hff = _outer(If, If)
        g_ = g * If                                    # pnqp.py:44-45
        H_ = H * Hff + eye                             # pnqp.py:46-48
        if n == 1:
            dx = -(1.0 / H_.squeeze(2)) * g_           # pnqp.py:51
        else:
            dx = -torch.linalg.solve(H_, g_.unsqueeze(2)).squeeze(2)
        J = torch.norm(dx, 2, 1) >= 1e-4               # pnqp.py:56
        if int(J.sum()) == 0:                          # pnqp.py:57-59
            return PnqpOut(x, H_, If, i, True)
        alpha = torch.ones(B, dtype=H.dtype)
        max_armijo = GAMMA
        count = 0
        while max_armijo <= GAMMA and count < 10:      # pnqp.py:65
            maybe_x = _clamp(x + alpha.unsqueeze(1) * dx, lower, upper)
            arm = torch.full((B,), GAMMA + 1e-6, dtype=H.dtype)
            ratio = (obj(x) - obj(maybe_x)) / _dot(g, x - maybe_x)
            arm[J] = ratio[J]                          # pnqp.py:71-72
            alpha[arm <= GAMMA] *= 0.1                 # pnqp.py:73-74
            max_armijo = torch.max(arm).item()
            count += 1
        x = maybe_x                                    # pnqp.py:78
    return PnqpOut(x, H_, If, n_iter - 1, False)       # pnqp.py:81-82


# --------------------------------------------------------------------------
# Riccati backward recursion  (lqr_step.py:52-160, lqr_step_backup.py:163-259)
# --------------------------------------------------------------------------
def lqr_backward(C, c, F, f, u, n_state, n_ctrl, u_lower=None, u_upper=None,
                 u_zero_I=None, gain_solve="pinv", delta_u=None):
    """Returns (Ks, ks, n_total_qp_iter); Ks/ks are lists in *reverse* time
    order exactly as the reference builds them (Ks[0] belongs to t=T-1).
    ``gain_solve``: "pinv" (lqr_step.py:88-94) or "chol_reg"
    (lqr_step_backup.py:202-205, Cholesky of Quu + 1e-6 I)."""
    T = C.shape[0]
    ns = n_state
    Ks, ks = [], []
    prev_k = None
    n_qp = 0
    V = v = None
    for t in range(T - 1, -1, -1):
        if t == T - 1:
            Q, qv = C[t], c[t]
        else:
            Ft = F[t]
            FtT = Ft.transpose(1, 2)
            Q = C[t] + FtT.bmm(V).bmm(Ft)              # lqr_step.py:68
            if f is None or f.nelement() == 0:
                qv = c[t] + _mv(FtT, v)                # lqr_step.py:70
            else:
                qv = c[t] + _mv(FtT.bmm(V), f[t]) + _mv(FtT, v)
        Qxx, Qxu = Q[:, :ns, :ns], Q[:, :ns, ns:]
        Qux, Quu = Q[:, ns:, :ns], Q[:, ns:, ns:]
        qx, qu = qv[:, :ns], qv[:, ns:]

        if u_lower is None:
            if n_ctrl == 1 and u_zero_I is None:       # lqr_step.py:84-86
                K = -(1.0 / Quu) * Qux
                k = -(1.0 / Quu.squeeze(2)) * qu
            elif u_zero_I is None:
                if gain_solve == "pinv":               # lqr_step.py:88-94
                    inv = torch.stack([torch.pinverse(Quu[i])
                                       for i in range(Quu.shape[0])])
                    K = -inv.bmm(Qux)
                    k = _mv(-inv, qu)
                else:                                  # lqr_step_backup.py:202-205
                    L = torch.linalg.cholesky(
                        Quu + 1e-6 * torch.eye(n_ctrl, dtype=Quu.dtype))
                    K = -torch.cholesky_solve(Qux, L)
                    k = -torch.cholesky_solve(qu.unsqueeze(2), L).squeeze(2)
            else:                                      # lqr_step.py:99-127
                I = u_zero_I[t].to(Quu.dtype)
                notI = 1 - I
                qu_ = qu * notI
                Quu_ = Quu * _outer(notI, notI)
                Quu_ = Quu_ + torch.diag_embed(I) * 1e-8
                Qux_ = Qux * notI.unsqueeze(2)
                if n_ctrl == 1:
                    K = -(1.0 / Quu_) * Qux_
                    k = -(1.0 / Quu.squeeze(2)) * qu_  # unmasked Quu (lqr_step.py:123)
                else:
                    K = -torch.linalg.solve(Quu_, Qux_)
                    k = -torch.linalg.solve(Quu_, qu_.unsqueeze(2)).squeeze(2)
        else:                                          # lqr_step.py:128-148
            lb = _bound(u_lower, t) - u[t]
            ub = _bound(u_upper, t) - u[t]
            if delta_u is not None:                    # lqr_step.py:132-134
                lb = torch.where(lb < -delta_u, torch.full_like(lb, -delta_u), lb)
                ub = torch.where(ub > delta_u, torch.full_like(ub, delta_u), ub)
            out = pnqp(Quu, qu, lb, ub, x_init=prev_k, n_iter=20)
            k = out.x
            n_qp += 1 + out.n_iter
            prev_k = k
            Qux_ = Qux * out.If.unsqueeze(2)
            if n_ctrl == 1:
                K = -((1.0 / out.Hfree) * Qux_)
            else:
                K = -torch.linalg.solve(out.Hfree, Qux_)
        KT = K.transpose(1, 2)
        Ks.append(K)
        ks.append(k)
        V = Qxx + Qxu.bmm(K) + KT.bmm(Qux) + KT.bmm(Quu).bmm(K)   # lqr_step.py:155
        v = qx + _mv(Qxu, k) + _mv(KT, qu) + _mv(KT.bmm(Quu), k)  # lqr_step.py:156-158
    return Ks, ks, n_qp


# --------------------------------------------------------------------------
# rollout, cost, line search  (util.py:104-153, lqr_step.py:164-261)
# --------------------------------------------------------------------------
def step_dynamics(dynamics, t, x, u):
    if isinstance(dynamics, LinDx):                    # util.py:117-121
        nx = _mv(dynamics.F[t], torch.cat((x, u), 1))
        if dynamics.f is not None and dynamics.f.nelement() > 0:
            nx = nx + dynamics.f[t]
        return nx
    return dynamics(x, u)


def get_traj(T, u, x_init, dynamics):                  # util.py:104-127
    x = [x_init]
    for t in range(T - 1):
        x.append(step_dynamics(dynamics, t, x[t], u[t]))
    return torch.stack(x, 0)


def get_cost(T, u, cost, x):                           # util.py:130-153
    objs = []
    for t in range(T):
        xut = torch.cat((x[t], u[t]), 1)
        objs.append(0.5 * _quad(xut, cost.C[t]) + _dot(xut, cost.c[t]))
    return torch.sum(torch.stack(objs, 0), dim=0)


LqrFwdOut = namedtuple("LqrFwdOut", "x u costs full_du_norm mean_alphas alphas n_ls")


def lqr_forward(x_init, cost, dynamics, Ks, ks, x, u, n_state, n_ctrl,
                u_lower=None, u_upper=None, u_zero_I=None,
                linesearch_decay=0.2, max_linesearch_iter=10, delta_u=None):
    """lqr_step.py:164-261.  Line search over the *true* dynamics."""
    T, B = u.shape[0], u.shape[1]
    old_cost = get_cost(T, u, cost, x)                 # lqr_step.py:169
    alphas = torch.ones(B, dtype=u.dtype)
    cur = None
    full_du = None
    i = 0
    while (cur is None or bool(torch.any(cur > old_cost))) and \
            i < max_linesearch_iter:
        new_u, new_x = [], [x_init]
        dx = torch.zeros_like(x_init)
        objs = []
        for t in range(T):
            K, k = Ks[T - 1 - t], ks[T - 1 - t]
            nxt = new_x[t]
            nu = _mv(K, dx) + u[t] + alphas.unsqueeze(1) * k   # lqr_step.py:192
            if u_zero_I is not None:
                nu = nu.clone()
                nu[u_zero_I[t]] = 0.0                  # lqr_step.py:197-198
            if u_lower is not None:
                lb, ub = _bound(u_lower, t), _bound(u_upper, t)
                if delta_u is not None:                # lqr_step.py:204-211
                    lo_t, hi_t = u[t] - delta_u, u[t] + delta_u
                    lb_l = lb if torch.is_tensor(lb) else torch.full_like(lo_t, lb)
                    ub_l = ub if torch.is_tensor(ub) else torch.full_like(hi_t, ub)
                    lb = torch.where(lo_t < lb_l, lb_l, lo_t)
                    ub = torch.where(hi_t > ub_l, ub_l, hi_t)
                nu = _clamp(nu, lb, ub)
            new_u.append(nu)
            xut = torch.cat((nxt, nu), 1)
            if t < T - 1:
                nx1 = step_dynamics(dynamics, t, nxt, nu)
                new_x.append(nx1)
                dx = nx1 - x[t + 1]                    # lqr_step.py:228
            objs.append(0.5 * _quad(xut, cost.C[t]) + _dot(xut, cost.c[t]))
        cur = torch.sum(torch.stack(objs), dim=0)
        new_u = torch.stack(new_u)
        new_x = torch.stack(new_x)
        if full_du is None:                            # lqr_step.py:243-245
            full_du = (u - new_u).transpose(1, 2).reshape(B, -1).norm(2, 1)
        alphas[cur > old_cost] *= linesearch_decay     # lqr_step.py:247
        i += 1
    alphas[cur > old_cost] /= linesearch_decay         # lqr_step.py:252
    return LqrFwdOut(new_x, new_u, cur, full_du, alphas.mean(), alphas, i)


def c_back(C, c, x, u):                                # lqr_step.py:289-295
    tau = torch.cat((x, u), 2)
    return torch.einsum("tbij,tbj->tbi", C, tau) + c


LqrStepOut = namedtuple(
    "LqrStepOut", "x u n_total_qp_iter costs full_du_norm mean_alphas Ks ks alphas")


def lqr_step(x_init, C, c, F, x, u, cost, dynamics, n_state, n_ctrl,
             u_lower=None, u_upper=None, u_zero_I=None, linesearch_decay=0.2,
             max_linesearch_iter=10, gain_solve="pinv", delta_u=None):
    """LQRStepFn.forward, lqr_step.py:277-309 (delta-space Taylor expansion,
    f_back=None)."""
    T = C.shape[0]
    cb = torch.stack([_mv(C[t], torch.cat((x[t], u[t]), 1)) + c[t]
                      for t in range(T)])
    Ks, ks, nqp = lqr_backward(C, cb, F, None, u, n_state, n_ctrl, u_lower,
                               u_upper, u_zero_I, gain_solve, delta_u)
    o = lqr_forward(x_init, cost, dynamics, Ks, ks, x, u, n_state, n_ctrl,
                    u_lower, u_upper, u_zero_I, linesearch_decay,
                    max_linesearch_iter, delta_u)
    return LqrStepOut(o.x, o.u, nqp, o.costs, o.full_du_norm, o.mean_alphas,
                      Ks, ks, o.alphas)


# --------------------------------------------------------------------------
# env_dx dynamics: forward + analytic first-order Jacobian
# --------------------------------------------------------------------------
class PendulumDx:
    """env_dx/pendulum.py:28-95 (simple=True) and get_linear_dyn 444-475."""
    n_state, n_ctrl = 3, 1
    dt = 0.05
    max_torque = 2.0
    lower, upper = -2.0, 2.0
    mpc_eps, linesearch_decay, max_linesearch_iter = 1e-3, 0.2, 5

    def __init__(self, params=None, dtype=torch.float32):
        self.params = (torch.tensor((10., 1., 1.), dtype=dtype)
                       if params is None else params)

    def get_true_obj(self):                            # pendulum.py:117-125
        dt = self.params.dtype
        gw = torch.tensor([1., 1., 0.1], dtype=dt)
        gs = torch.tensor([1., 0., 0.], dtype=dt)
        q = torch.cat((gw, 0.001 * torch.ones(1, dtype=dt)))
        p = torch.cat((-torch.sqrt(gw) * gs, torch.zeros(1, dtype=dt)))
        return q, p

    def __call__(self, x, u):                          # pendulum.py:60-95
        g, m, l = torch.unbind(self.params.detach())
        uc = torch.clamp(u, -self.max_torque, self.max_torque)[:, 0]
        c, s, w = torch.unbind(x, dim=1)
        th = torch.atan2(s, c)
        nw = w + self.dt * (-3. * g / (2. * l) * (-s) + 3. * uc / (m * l ** 2))
        nth = th + nw * self.dt
        return torch.stack((torch.cos(nth), torch.sin(nth), nw), dim=1)

    def get_linear_dyn(self, x, u):                    # pendulum.py:444-475
        g, m, l = torch.unbind(self.params.detach())
        dt = self.dt
        c, s, w = x[:, 0], x[:, 1], x[:, 2]
        uu = u[:, 0]
        phi = dt * (dt * (3 * g * s / (2 * l) + 3 * uu / (l ** 2 * m)) + w) \
            + torch.atan2(s, c)
        sp, cp = torch.sin(phi), torch.cos(phi)
        r2 = c ** 2 + s ** 2
        a = 3 * dt ** 2 * g / (2 * l)
        b = 3 * dt ** 2 / (l ** 2 * m)
        z, o = torch.zeros_like(c), torch.ones_like(c)
        rows = [
            [s * sp / r2, -(c / r2 + a) * sp, -dt * sp, -b * sp],
            [-s * cp / r2, (c / r2 + a) * cp, dt * cp, b * cp],
            [z, o * (3 * dt * g / (2 * l)), o, o * (3 * dt / (l ** 2 * m))],
        ]
        return torch.stack([torch.stack(r, 1) for r in rows], 1)


class CartpoleDx:
    """env_dx/cartpole.py:29-97 and get_linear_dyn 790-839."""
    n_state, n_ctrl = 5, 1
    dt = 0.05
    force_mag = 100.0
    lower, upper = -100.0, 100.0
    mpc_eps, linesearch_decay, max_linesearch_iter = 1e-4, 0.5, 2

    def __init__(self, params=None, dtype=torch.float32):
        self.params = (torch.tensor((9.8, 1.0, 0.1, 0.5), dtype=dtype)
                       if params is None else params)

    def get_true_obj(self):                            # cartpole.py:859-867
        dt = self.params.dtype
        gw = torch.tensor([0.1, 0.1, 1., 1., 0.1], dtype=dt)
        gs = torch.tensor([0., 0., 1., 0., 0.], dtype=dt)
        q = torch.cat((gw, 0.001 * torch.ones(1, dtype=dt)))
        p = torch.cat((-torch.sqrt(gw) * gs, torch.zeros(1, dtype=dt)))
        return q, p

    def __call__(self, state, u):                      # cartpole.py:64-97
        g, mc, mp, l = torch.unbind(self.params.detach())
        M = mp + mc
        pml = mp * l
        uc = torch.clamp(u[:, 0], -self.force_mag, self.force_mag)
        x, dx, c, s, w = torch.unbind(state, dim=1)
        th = torch.atan2(s, c)
        cart_in = (uc + pml * w ** 2 * s) / M
        th_acc = (g * s - c * cart_in) / (l * (4. / 3. - mp * c ** 2 / M))
        xacc = cart_in - pml * th_acc * c / M
        nx = x + self.dt * dx
        ndx = dx + self.dt * xacc
        nth = th + self.dt * w
        nw = w + self.dt * th_acc
        return torch.stack((nx, ndx, torch.cos(nth), torch.sin(nth), nw), 1)

    def get_linear_dyn(self, x, u):                    # cartpole.py:790-839
        """Closed-form Jacobian of the Euler step wrt (x, dx, cos, sin, dth, u),
        ignoring the input clamp (the reference does the same)."""
        g, mc, mp, l = torch.unbind(self.params.detach())
        dt = self.dt
        M = mc + mp
        c, s, w = x[:, 2], x[:, 3], x[:, 4]
        uu = u[:, 0]
        z, o = torch.zeros_like(c), torch.ones_like(c)
        A = w ** 2 * l * mp * s + uu                   # cart force numerator
        G = -c * A / M + g * s                         # th_acc numerator
        den = -c ** 2 * mp / M + 4. / 3.               # 4/3 - mp c^2 / M
        den2 = (-3 * c ** 2 * mp / (4 * M) + 1) ** 2   # (3/4 den)^2
        phi = dt * w + torch.atan2(s, c)
        sp, cp = torch.sin(phi), torch.cos(phi)
        r2 = c ** 2 + s ** 2
        # d(xacc)/d(c,s,w,u)
        xa_c = (-9 * c ** 2 * mp ** 2 * G / (8 * M ** 2 * den2)
                + c * mp * A / (M ** 2 * den) - mp * G / (M * den))
        xa_s = -c * mp * (-c * w ** 2 * l * mp / M + g) / (M * den) \
            + w ** 2 * l * mp / M
        xa_w = 2 * c ** 2 * w * l * mp ** 2 * s / (M ** 2 * den) \
            + 2 * w * l * mp * s / M
        xa_u = c ** 2 * mp / (M ** 2 * den) + 1 / M
        # dt * d(th_acc)/d(c,s,w,u)
        ta_c = 9 * c * dt * mp * G / (8 * l * M * den2) - dt * A / (l * M * den)
        ta_s = dt * (-c * w ** 2 * l * mp / M + g) / (l * den)
        ta_w = -2 * c * dt * w * mp * s / (M * den) + 1
        ta_u = -c * dt / (l * M * den)
        rows = [
            [o, o * dt, z, z, z, z],
            [z, o, dt * xa_c, dt * xa_s, dt * xa_w, dt * xa_u],
            [z, z, s * sp / r2, -c * sp / r2, -dt * sp, z],
            [z, z, -s * cp / r2, c * cp / r2, dt * cp, z],
            [z, z, ta_c, ta_s, ta_w, ta_u],
        ]
        return torch.stack([torch.stack(r, 1) for r in rows], 1)


def linearize_dynamics(x, u, dynamics):
    """mpc_explicit.py:516-546 (ANALYTIC): F_t = D(x_t,u_t), f_t = f(x_t,u_t)
    - D tau_t for t < T-1."""
    T, B, ns = x.shape
    nc = u.shape[2]
    _x = x[:-1].reshape(-1, ns)
    _u = u[:-1].reshape(-1, nc)
    new_x = dynamics(_x, _u)
    D = dynamics.get_linear_dyn(_x, _u)
    d = new_x - torch.einsum("bnm,bm->bn", D, torch.cat((_x, _u), -1))
    return D.reshape(T - 1, B, ns, ns + nc), d.reshape(T - 1, B, ns)


# --------------------------------------------------------------------------
# iLQR outer loop  (mpc.py:184-337 / mpc_explicit.py:182-358)
# --------------------------------------------------------------------------
MpcOut = namedtuple(
    "MpcOut", "x u costs full_du_norm n_iters F f Ks qp_iters converged log")


def mpc_forward(x_init, cost, dynamics, n_state, n_ctrl, T, u_lower=None,
                u_upper=None, u_zero_I=None, u_init=None, lqr_iter=10,
                eps=1e-7, linesearch_decay=0.2, max_linesearch_iter=10,
                not_improved_lim=5, best_cost_eps=1e-4, gain_solve="pinv",
                final_pass=True, delta_u=None):
    """MPC.forward (mpc.py:184-337).  ``cost`` is a QuadCost with dense
    C[T,B,n,n], c[T,B,n]; ``dynamics`` a LinDx or an env object with
    __call__/get_linear_dyn.  Returns best iterate, costs, and (for the
    backward passes) the final linearisation F, f and the gains of the final
    no-op LQR step (lqr_step_explicit.py:604-623)."""
    B = x_init.shape[0]
    dtype = x_init.dtype
    if u_init is None:
        u = torch.zeros(T, B, n_ctrl, dtype=dtype)     # mpc.py:230-231
    else:
        u = u_init.clone()
        if u.ndimension() == 2:
            u = u.unsqueeze(1).expand(T, B, -1).clone()
    best = None
    n_not_improved = 0
    log = []
    it = 0
    for it in range(lqr_iter):                         # mpc.py:248
        x = get_traj(T, u, x_init, dynamics)           # mpc.py:251
        if isinstance(dynamics, LinDx):
            F = dynamics.F
        else:
            F, _ = linearize_dynamics(x, u, dynamics)
        o = lqr_step(x_init, cost.C, cost.c, F, x, u, cost, dynamics, n_state,
                     n_ctrl, u_lower, u_upper, u_zero_I, linesearch_decay,
                     max_linesearch_iter, gain_solve, delta_u)
        x, u = o.x, o.u
        n_not_improved += 1                            # mpc.py:266
        if best is None:                               # mpc.py:271-277
            best = {"x": x.clone(), "u": u.clone(), "costs": o.costs.clone(),
                    "du": o.full_du_norm.clone()}
        else:                                          # mpc.py:278-285
            imp = o.costs <= best["costs"] + best_cost_eps
            if bool(imp.any()):
                n_not_improved = 0
            best["x"][:, imp] = x[:, imp]
            best["u"][:, imp] = u[:, imp]
            best["costs"][imp] = o.costs[imp]
            best["du"][imp] = o.full_du_norm[imp]
        log.append((o.n_total_qp_iter, float(o.full_du_norm.max()),
                    float(o.mean_alphas), float(best["costs"].mean())))
        if float(o.full_du_norm.max()) < eps or \
                n_not_improved > not_improved_lim:     # mpc.py:299-301
            break
    x, u = best["x"], best["u"]
    F = f = Ks = None
    if final_pass:
        if isinstance(dynamics, LinDx):
            F, f = dynamics.F, dynamics.f
        else:
            F, f = linearize_dynamics(x, u, dynamics)  # mpc.py:310 (diff=True)
        cb = c_back(cost.C, cost.c, x, u)
        Ks, _, _ = lqr_backward(cost.C, cb, F, None, u, n_state, n_ctrl,
                                u_lower, u_upper, u_zero_I, gain_solve)
        Ks = torch.stack(Ks, 0)     # reverse time order, lqr_step_explicit.py:617-618
    conv = bool(best["du"].max() <= eps)
    return MpcOut(x, u, best["costs"], best["du"], it + 1, F, f, Ks,
                  [l[0] for l in log], conv, log)


# --------------------------------------------------------------------------
# KKT / adjoint-LQR backward  (lqr_step.py:312-407)
# --------------------------------------------------------------------------
KktOut = namedtuple("KktOut", "dx_init dC dc dF df dx du")


def kkt_backward(dl_dx, dl_du, x_init, C, c, F, f, x, u, n_state, n_ctrl,
                 u_lower=None, u_upper=None, gain_solve="pinv",
                 want_df=True):
    """Gradients of a loss wrt (x_init, C, c, F, f) given dl/dx*, dl/du* at an
    LQR solution (x*, u*) = argmin of the box-constrained LQR (C,c,F,f).
    Restates LQRStepFn.backward, lqr_step.py:312-407: one adjoint LQR solve
    (``MPC(lqr_iter=1, u_zero_I=active set)`` on cost (C,-r), dynamics
    LinDx(F,None), x_init=0) followed by the two costate recursions."""
    T, B = x.shape[0], x.shape[1]
    ns = n_state
    r = torch.cat((dl_dx, dl_du), 2)                   # lqr_step.py:316-320
    if u_lower is None:
        I = None
    else:                                              # lqr_step.py:325-326
        I = (torch.abs(u - u_lower) <= 1e-8) | (torch.abs(u - u_upper) <= 1e-8)
    zero = torch.zeros_like(x_init)
    o = mpc_forward(zero, QuadCost(C, -r), LinDx(F, None), n_state, n_ctrl, T,
                    u_zero_I=I, lqr_iter=1, gain_solve=gain_solve,
                    final_pass=False)                  # lqr_step.py:328-340
    dx, du = o.x, o.u
    dxu = torch.cat((dx, du), 2)
    xu = torch.cat((x, u), 2)
    dC = -0.5 * (torch.einsum("tbi,tbj->tbij", dxu, xu)
                 + torch.einsum("tbi,tbj->tbij", xu, dxu))   # lqr_step.py:346-351
    dc = -dxu                                          # lqr_step.py:353
    lams = [None] * T
    dlams = [None] * T
    prev = dprev = None
    for t in range(T - 1, -1, -1):                     # lqr_step.py:355-385
        Cxx, Cxu = C[t, :, :ns, :ns], C[t, :, :ns, ns:]
        lam = _mv(Cxx, x[t]) + _mv(Cxu, u[t]) + c[t, :, :ns]
        dlam = _mv(Cxx, dx[t]) + _mv(Cxu, du[t]) - r[t, :, :ns]
        if prev is not None:
            FxT = F[t, :, :, :ns].transpose(1, 2)
            lam = lam + _mv(FxT, prev)
            dlam = dlam + _mv(FxT, dprev)
        lams[t], dlams[t] = lam, dlam
        prev, dprev = lam, dlam
    dF = torch.zeros_like(F)
    for t in range(T - 1):                             # lqr_step.py:387-395
        dF[t] = -(_outer(dlams[t + 1], xu[t]) + _outer(lams[t + 1], dxu[t]))
    dlams = torch.stack(dlams)
    df = -dlams[1:] if want_df else None               # lqr_step.py:397-402
    dx_init = -dlams[0]                                # lqr_step.py:404
    return KktOut(dx_init, dC, dc, dF, df, dx, du)


# --------------------------------------------------------------------------
# DiLQR implicit gradient (lqr_step_explicit.py:652-712 + fix_point_equ 458-598)
# in its algebraically identical matrix-free form (SURVEY Appendix C)
# --------------------------------------------------------------------------
def env_tables(dynamics, x, u):
    """get_matrices (cartpole.py:105-716 / pendulum.py:152-382), generated."""
    import env_tables_gen as G
    fn = (G.cartpole_tables if isinstance(dynamics, CartpoleDx) else
          G.rocket_tables if isinstance(dynamics, RocketDx) else G.pendulum_tables)
    return fn(x, u, dynamics.params.detach())


def grad_input(dynamics, X, U, K):
    """Closed-loop parameter-sensitivity rollout, cartpole.py:717-788 /
    pendulum.py:383-443.  ``K`` is indexed exactly like the reference does
    (K[t] of the *reverse-time* stack, SURVEY 8a-10 quirk)."""
    T, B, ns = X.shape
    nc = U.shape[2]
    n = ns + nc
    D, Dth, Dx, Du, xth, xx, xu = env_tables(dynamics, X.reshape(T * B, ns), U.reshape(T * B, nc))
    nth = Dth.shape[-1]
    D = D.reshape(T, B, ns, n)
    Dth = Dth.reshape(T, B, ns, n, nth)
    Dx = Dx.reshape(T, B, ns, n, ns)
    Du = Du.reshape(T, B, ns, n, nc)
    xth = xth.reshape(T, B, ns, nth)
    xx = xx.reshape(T, B, ns, ns)
    xu = xu.reshape(T, B, ns, nc)
    XU = torch.cat((X, U), -1)
    d_x = torch.einsum("tbnmk,tbm->tbnk", -Dx, XU)       # cartpole.py:752
    d_u = torch.einsum("tbnmk,tbm->tbnk", -Du, XU)       # cartpole.py:753
    G = torch.zeros(B, ns, nth, dtype=X.dtype)
    grad_D, grad_d = [], []
    Gm1 = None
    for t in range(T):
        Kt = K[t]
        if t > 0:
            Ktm1 = K[t - 1]
            Gm1 = G
            G = xth[t] + torch.matmul(xx[t] + torch.matmul(xu[t], Ktm1), G)   # :768
        if t < T - 1:                                                         # :773-775
            gD = Dth[t] + torch.matmul(Dx[t] + torch.matmul(Du[t], Kt.unsqueeze(1)),
                                       G.unsqueeze(1))
            grad_D.append(gD)
        if t > 0:                                                             # :778-782
            Z = torch.cat((Gm1, torch.matmul(Ktm1, Gm1)), 1)
            gd = G - torch.einsum("bnmk,bm->bnk", grad_D[t - 1], XU[t - 1]) \
                - torch.matmul(D[t - 1], Z)
            grad_d.append(gd)
    return (torch.stack(grad_D), torch.stack(grad_d), Dx[:T - 1], Du[:T - 1], D[:T - 1],
            d_x[:T - 1], d_u[:T - 1])


DilqrOut = namedtuple("DilqrOut", "dC dc dtheta w n_passes resid")


def dilqr_backward(dl_dx, dl_du, x_init, C, c, x, u, dynamics, n_state, n_ctrl,
                   u_lower=None, u_upper=None, n_passes=8, tol=None):
    """Implicit (fixed-point) gradient of lqr_step_explicit.LQRStepFn.backward:
       solve A' w = g with A = I - (J_F dD/dtau + J_f dd/dtau) by Richardson
       iteration w <- g + M' w, where M' w needs one KKT adjoint pass; then one
       more KKT pass with r = w gives dC, dc and (dF_w, df_w), and
       dtheta_b = <dF_w, dD/dtheta> + <df_w, dd/dtheta>.
    The adjoint solves use mpc_backup/lqr_step_backup (Cholesky + 1e-6 I when
    unconstrained, lqr_step_explicit.py:277-290)."""
    T, B = x.shape[0], x.shape[1]
    F, f = linearize_dynamics(x, u, dynamics)
    cb = c_back(C, c, x, u)
    Ks, _, _ = lqr_backward(C, cb, F, None, u, n_state, n_ctrl, u_lower, u_upper)
    Ks = torch.stack(Ks, 0)                                   # reverse-time stack (:617-618)
    grad_D, grad_d, Dx, Du, D, d_x, d_u = grad_input(dynamics, x, u, Ks)
    g = torch.cat((dl_dx, dl_du), 2)
    w = g.clone()
    resid = None
    k = None
    passes = 0
    for it in range(n_passes + 1):
        k = kkt_backward(w[:, :, :n_state], w[:, :, n_state:], x_init, C, c, F, f, x, u,
                         n_state, n_ctrl, u_lower, u_upper, gain_solve="chol_reg")
        if it == n_passes:
            break
        Mw = torch.zeros_like(g)
        Mw[:T - 1, :, :n_state] = torch.einsum("tbnm,tbnmk->tbk", k.dF, Dx) + \
            torch.einsum("tbn,tbnk->tbk", k.df, d_x)
        Mw[:T - 1, :, n_state:] = torch.einsum("tbnm,tbnmk->tbk", k.dF, Du) + \
            torch.einsum("tbn,tbnk->tbk", k.df, d_u)
        w_new = g + Mw
        resid = float((w_new - w).abs().max() / (w_new.abs().max() + 1e-300))
        w = w_new
        passes = it + 1
        if tol is not None and resid < tol:
            k = kkt_backward(w[:, :, :n_state], w[:, :, n_state:], x_init, C, c, F, f, x, u,
                             n_state, n_ctrl, u_lower, u_upper, gain_solve="chol_reg")
            break
    dtheta = torch.einsum("tbnm,tbnmk->bk", k.dF, grad_D) + \
        torch.einsum("tbn,tbnk->bk", k.df, grad_d)
    return DilqrOut(k.dC, k.dc, dtheta, w, passes, resid)


class RocketDx:
    """env_dx/rocket.py:14-164 (6-DoF rocket, quaternion attitude) and its analytic
    Jacobian get_linear_dyn 324-426.  State r(3), v(3), q(4), w(3); control thrust
    (3); params (Jx, Jy, Jz, mass, l), dt = 0.1.  Mirrors the reference's quirk of
    returning the UN-normalised quaternion (rocket.py:158-164)."""
    n_state, n_ctrl = 13, 3
    dt = 0.1
    max_thrust = 400.0
    lower, upper = -20.0, 20.0          # SURVEY 8d config 3 (float bounds)
    mpc_eps, linesearch_decay, max_linesearch_iter = 1e-3, 0.2, 5

    def __init__(self, params=None, dtype=torch.float32):
        self.params = (torch.tensor((0.5, 1.0, 1.0, 1.0, 1.0), dtype=dtype)
                       if params is None else params)

    def get_true_obj(self):                            # rocket.py:212-232
        dt = self.params.dtype
        gw = torch.ones(13, dtype=dt)
        gw[0:3] = 10.0
        gw[6:10] = 0.1
        gs = torch.zeros(13, dtype=dt)
        gs[6] = 1.0
        cp = torch.tensor([1.0, 1.0, 0.4], dtype=dt)
        tilt_Q = 50.0 * torch.tensor([0., 0., 4., 4.], dtype=dt)
        q = torch.cat((gw, cp))
        q[6:10] = tilt_Q * 50.0                        # tilt_penalty applied twice (:74-77,225)
        px = -torch.sqrt(gw) * gs
        px[6:10] = 0.0
        p = torch.cat((px, torch.zeros(3, dtype=dt)))
        return q, p

    def __call__(self, x, u):                          # rocket.py:82-164
        Jx, Jy, Jz, mass, l = torch.unbind(self.params.detach())
        v, q, w = x[:, 3:6], x[:, 6:10], x[:, 10:13]
        T_B = torch.clamp(u, -self.max_thrust, self.max_thrust)
        q0, q1, q2, q3 = q.unbind(-1)
        C_B_I = torch.stack([
            torch.stack([1 - 2 * (q2 ** 2 + q3 ** 2), 2 * (q1 * q2 + q0 * q3), 2 * (q1 * q3 - q0 * q2)], -1),
            torch.stack([2 * (q1 * q2 - q0 * q3), 1 - 2 * (q1 ** 2 + q3 ** 2), 2 * (q2 * q3 + q0 * q1)], -1),
            torch.stack([2 * (q1 * q3 + q0 * q2), 2 * (q2 * q3 - q0 * q1), 1 - 2 * (q1 ** 2 + q2 ** 2)], -1),
        ], 1)
        tg = torch.bmm(C_B_I.transpose(1, 2), T_B.unsqueeze(-1)).squeeze(-1)
        g = torch.tensor([-10., 0., 0.], dtype=x.dtype).expand(x.shape[0], 3)
        dv = tg / mass + g
        wx, wy, wz = w.unbind(-1)
        z = torch.zeros_like(wx)
        om = torch.stack([
            torch.stack([z, -wx, -wy, -wz], -1), torch.stack([wx, z, wz, -wy], -1),
            torch.stack([wy, -wz, z, wx], -1), torch.stack([wz, wy, -wx, z], -1)], 1)
        dq = 0.5 * torch.bmm(om, q.unsqueeze(-1)).squeeze(-1)
        rT = torch.stack([-l / 2, torch.zeros_like(l), torch.zeros_like(l)]).to(x.dtype).expand(x.shape[0], 3)
        torque = torch.linalg.cross(rT, T_B, dim=1)
        J = torch.stack([Jx, Jy, Jz]).to(x.dtype)
        Jw = w * J
        dw = (1.0 / J) * (torque - torch.linalg.cross(w, Jw, dim=1))
        deriv = torch.cat([v, dv, dq, dw], 1)
        return x + deriv * self.dt

    def get_linear_dyn(self, x, u):                    # rocket.py:324-426
        import env_tables_gen as G
        return G.rocket_tables(x, u, self.params.detach())[0]


# ---------------------------------------------------------------------------
# Closed-loop expert data (il_env.py:57-79, 96-151)
# ---------------------------------------------------------------------------
def sample_xinit(env, n_batch):                        # il_env.py:57-79
    import math

    def uniform(shape, low, high):
        return torch.rand(shape) * (high - low) + low

    if env == "pendulum":
        th = uniform(n_batch, -(1 / 2) * math.pi, (1 / 2) * math.pi)
        thdot = uniform(n_batch, -1., 1.)
        return torch.stack((torch.cos(th), torch.sin(th), thdot), dim=1)
    assert env == "cartpole"
    x = uniform(n_batch, -0.5, 0.5) * 0
    dx = uniform(n_batch, -0.5, 0.5) * 0
    th = uniform(n_batch, -math.pi, math.pi) * 0 + torch.ones(n_batch) * 3.1415926 / 1.05
    dth = uniform(n_batch, -1., 1.) * 0
    return torch.stack((x, dx, torch.cos(th), torch.sin(th), dth), dim=1)


def closed_loop(dynamics, x_init_all, T, lqr_iter):
    """populate_data2 (il_env.py:96-151): for every sample, T receding-horizon MPC
    calls with n_batch = 1; apply the first control, shift the warm start."""
    q, p = dynamics.get_true_obj()
    n = q.shape[0]
    dtype = x_init_all.dtype
    Q = torch.diag(q.to(dtype)).reshape(1, 1, n, n).repeat(T, 1, 1, 1)
    pp = p.to(dtype).reshape(1, 1, n).repeat(T, 1, 1)
    taus = []
    for i in range(x_init_all.shape[0]):
        x = x_init_all[i].unsqueeze(0)
        u_init = None
        xs, us = [x.squeeze(0)], []
        for _ in range(T):
            o = mpc_forward(x, QuadCost(Q.clone(), pp.clone()), dynamics, dynamics.n_state,
                            dynamics.n_ctrl, T, u_lower=dynamics.lower, u_upper=dynamics.upper,
                            u_init=u_init, lqr_iter=lqr_iter, eps=dynamics.mpc_eps,
                            linesearch_decay=dynamics.linesearch_decay,
                            max_linesearch_iter=dynamics.max_linesearch_iter,
                            final_pass=False)
            a = o.u[0]
            us.append(a.squeeze(0))
            x = dynamics(x, a)
            xs.append(x.squeeze(0))
            u_init = torch.cat((o.u[1:], torch.zeros(1, 1, dynamics.n_ctrl, dtype=dtype)), 0)
            u_init[-2] = u_init[-3]
        taus.append(torch.cat((torch.stack(xs[:-1]), torch.stack(us)), 1))
    return torch.stack(taus)


# ---------------------------------------------------------------------------
# dynamics.NNDynamics (dynamics.py:15-130), one hidden layer, as an oracle dynamics
# object for mpc_forward (same protocol as the env classes: __call__ / get_linear_dyn)
# ---------------------------------------------------------------------------
class NNDynamics:
    def __init__(self, W1, b1, W2, b2, activation="sigmoid", passthrough=True):
        self.W1, self.b1, self.W2, self.b2 = W1, b1, W2, b2
        self.activation, self.passthrough = activation, passthrough
        self.n_state = W2.shape[0]
        self.n_ctrl = W1.shape[1] - self.n_state

    def _hidden(self, x, u):
        a = torch.cat((x, u), 1) @ self.W1.t() + self.b1          # dynamics.py:66-68
        return torch.sigmoid(a) if self.activation == "sigmoid" else torch.relu(a)

    def __call__(self, x, u):                                    # dynamics.py:57-79
        z = self._hidden(x, u) @ self.W2.t() + self.b2
        return z + x if self.passthrough else z

    def get_linear_dyn(self, x, u):                              # grad_input, :81-130
        z = self._hidden(x, u)
        d = z * (1. - z) if self.activation == "sigmoid" else (z > 0.).to(z.dtype)
        J = self.W2.unsqueeze(0).expand(x.shape[0], -1, -1).bmm(self.W1.unsqueeze(0) * d.unsqueeze(2))
        if self.passthrough:
            J = J.clone()
            J[:, :, :self.n_state] += torch.eye(self.n_state, dtype=J.dtype)
        return J
