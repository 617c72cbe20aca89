"""``MPC`` -- drop-in for the reference's ``mpc.MPC`` (mpc.py:58-337): same
constructor, same ``forward(x_init, cost, dx) -> (x, u, costs)``, gradients by
the KKT / adjoint-LQR backward of ``LQRStepFn.backward`` (lqr_step.py:312-407).

All arithmetic runs in the sm_100a kernels behind ``libdilqr.so``; this module
is the host-side mirror of the reference interface (argument handling, the
stop rule, warnings, unconverged masking).
"""
import sys
from enum import Enum

import torch
from torch import nn
from torch.autograd import Function

from . import _lib, _solver
from .definitions import QuadCost, LinDx
from .dynamics import AffineDynamics, NNDynamics


class GradMethods(Enum):          # mpc.py:29-33
    AUTO_DIFF = 1
    FINITE_DIFF = 2
    ANALYTIC = 3
    ANALYTIC_CHECK = 4


def _dyn_spec(dx):
    if isinstance(dx, LinDx):
        return _solver.DynSpec(_lib.DYN_LINDX, F=dx.F, f=dx.f)
    kind = getattr(dx, "_dilqr_kind", None)
    if kind is None:
        raise NotImplementedError(
            "dynamics of type %s: only LinDx and the env_dx models of this package "
            "(analytic linearisation) are supported" % type(dx).__name__)
    params = dx._theta_list() if hasattr(dx, "_theta_list") else dx.params.detach().double().cpu().tolist()
    return _solver.DynSpec(kind, params=params)


class _MPCFn(Function):
    """Forward: fused iLQR solve.  Backward: KKT adjoint (lqr_step.py:312-407)."""

    @staticmethod
    def forward(ctx, mod, dx, x_init, C, c, F, f):
        dyn = _dyn_spec(dx)
        x, u, costs, info = _solver.solve_mpc(
            x_init, C, c, dyn, mod.n_state, mod.n_ctrl, mod.T,
            u_lower=mod.u_lower, u_upper=mod.u_upper, u_zero_I=mod.u_zero_I,
            u_init=mod.u_init, lqr_iter=mod.lqr_iter, eps=mod.eps,
            linesearch_decay=mod.linesearch_decay,
            max_linesearch_iter=mod.max_linesearch_iter,
            not_improved_lim=mod.not_improved_lim, best_cost_eps=mod.best_cost_eps,
            gain_solve=mod._gain_solve, solo=mod.solo, verbose=mod.verbose, delta_u=mod.delta_u)
        mod.last_info = info
        ctx.mod = mod
        ctx.dyn_kind = dyn.kind
        ctx.mask = None
        eps_cmp = float(torch.tensor(mod.eps, dtype=x.dtype))
        if mod.detach_unconverged:                       # mpc.py:321-334
            # full_du_norm of the best iterates decides convergence
            if float(info.full_du_norm.max()) > eps_cmp:
                if mod.exit_unconverged:
                    assert False
                if mod.verbose >= 0:
                    print("LQR Warning: All examples did not converge to a fixed point.")
                    print("Detaching and *not* backpropping through the bad examples.")
                ctx.mask = (info.full_du_norm < eps_cmp).to(x.dtype)
        ctx.save_for_backward(x_init, C, c, F if F is not None else x.new_empty(0),
                              f if f is not None else x.new_empty(0), x, u)
        ctx.mark_non_differentiable(costs)
        return x, u, costs

    @staticmethod
    def backward(ctx, dl_dx, dl_du, _dcosts):
        mod = ctx.mod
        x_init, C, c, F, f, x, u = ctx.saved_tensors
        if ctx.dyn_kind != _lib.DYN_LINDX:
            raise NotImplementedError(
                "mpc.MPC differentiates LinDx problems (KKT gradients); use "
                "mpc_explicit.MPC for env_dx dynamics")
        if ctx.mask is not None:
            dl_dx = dl_dx * ctx.mask.view(1, -1, 1)
            dl_du = dl_du * ctx.mask.view(1, -1, 1)
        dx0, dC, dc, dF, df = _solver.kkt_backward(
            dl_dx.contiguous(), dl_du.contiguous(), x_init, C, c, F, f, x, u,
            mod.n_state, mod.n_ctrl, mod.u_lower, mod.u_upper,
            gain_solve=mod._gain_solve, back_eps=mod.back_eps)
        if f.nelement() == 0:
            df = None
        return None, None, dx0, dC, dc, dF, df


class _KKTAtSolutionFn(Function):
    """The final no-op LQR step of the reference (mpc.py:314-315, lqr_step.py:278-282):
    forward hands back the solution, backward is the KKT adjoint of the LQR subproblem
    linearised there -- gradients wrt x_init, C, c AND the linearisation F, f, through
    which autograd reaches the parameters of a Module dynamics."""

    @staticmethod
    def forward(ctx, mod, mask, x_init, C, c, F, f, x, u):
        ctx.mod, ctx.mask = mod, mask
        ctx.save_for_backward(x_init, C, c, F, f, x, u)
        return x.clone(), u.clone()

    @staticmethod
    def backward(ctx, dl_dx, dl_du):
        mod = ctx.mod
        x_init, C, c, F, f, x, u = ctx.saved_tensors
        if ctx.mask is not None:
            dl_dx = dl_dx * ctx.mask.view(1, -1, 1)
            dl_du = dl_du * ctx.mask.view(1, -1, 1)
        dx0, dC, dc, dF, df = _solver.kkt_backward(
            dl_dx.contiguous(), dl_du.contiguous(), x_init, C, c, F, f, x, u,
            mod.n_state, mod.n_ctrl, mod.u_lower, mod.u_upper,
            gain_solve=mod._gain_solve, back_eps=mod.back_eps)
        return None, None, dx0, dC, dc, dF, df, None, None


class MPC(nn.Module):
    """See the reference docstring (mpc.py:59-121); arguments are identical."""

    _gain_solve = _lib.GAIN_PLAIN     # lqr_step.py:88-94
    _Fn = _MPCFn

    def __init__(self, n_state, n_ctrl, T, u_lower=None, u_upper=None, u_zero_I=None,
                 u_init=None, lqr_iter=10, grad_method=GradMethods.ANALYTIC, delta_u=None,
                 verbose=0, eps=1e-7, back_eps=1e-7, n_batch=None, linesearch_decay=0.2,
                 max_linesearch_iter=10, exit_unconverged=True, detach_unconverged=True,
                 backprop=True, slew_rate_penalty=None, prev_ctrl=None,
                 not_improved_lim=5, best_cost_eps=1e-4, solo=False):
        super().__init__()
        assert (u_lower is None) == (u_upper is None)      # mpc.py:146
        assert max_linesearch_iter > 0                     # mpc.py:147
        self.n_state, self.n_ctrl, self.T = n_state, n_ctrl, T
        det = lambda v: v if (v is None or isinstance(v, float)) else v.detach()
        self.u_lower, self.u_upper = det(u_lower), det(u_upper)
        self.u_zero_I = None if u_zero_I is None else u_zero_I.detach()
        self.u_init = None if u_init is None else u_init.detach()
        self.lqr_iter = lqr_iter
        self.grad_method = grad_method
        self.delta_u = delta_u
        self.verbose = verbose
        self.eps, self.back_eps = eps, back_eps
        self.n_batch = n_batch
        self.linesearch_decay = linesearch_decay
        self.max_linesearch_iter = max_linesearch_iter
        self.exit_unconverged = exit_unconverged
        self.detach_unconverged = detach_unconverged
        self.backprop = backprop
        self.not_improved_lim = not_improved_lim
        self.best_cost_eps = best_cost_eps
        self.slew_rate_penalty = slew_rate_penalty
        self.prev_ctrl = prev_ctrl
        self.solo = solo
        self.last_info = None

    def _expand_cost(self, cost, n_batch):
        """mpc.py:205-226: accept C[n,n] / C[T,n,n] / C[T,B,n,n] and c likewise."""
        n = self.n_state + self.n_ctrl
        C, c = cost
        if C.ndimension() == 2:
            C = C.unsqueeze(0).unsqueeze(0).expand(self.T, n_batch, n, -1)
        elif C.ndimension() == 3:
            C = C.unsqueeze(1).expand(self.T, n_batch, n, -1)
        if c.ndimension() == 1:
            c = c.unsqueeze(0).unsqueeze(0).expand(self.T, n_batch, -1)
        elif c.ndimension() == 2:
            c = c.unsqueeze(1).expand(self.T, n_batch, -1)
        if C.ndimension() != 4 or c.ndimension() != 3:
            print('MPC Error: Unexpected QuadCost shape.')
            sys.exit(-1)
        return C, c

    def forward(self, x_init, cost, dx):
        quad = isinstance(cost, QuadCost)
        if not quad and not isinstance(cost, nn.Module):
            raise TypeError("cost must be a QuadCost or an nn.Module (mpc.py:447-487)")
        if self.n_batch is not None:
            n_batch = self.n_batch
        elif quad and cost.C.ndimension() == 4:
            n_batch = cost.C.size(1)
        else:
            print('MPC Error: Could not infer batch size, pass in as n_batch')
            sys.exit(-1)
        assert x_init.ndimension() == 2 and x_init.size(0) == n_batch
        if isinstance(dx, AffineDynamics):      # time-invariant LinDx (dynamics.py:159-202)
            dx = LinDx(*dx.as_lindx(self.T, n_batch, x_init.dtype, x_init.device))
        generic_dx = not isinstance(dx, (LinDx, NNDynamics)) and getattr(dx, "_dilqr_kind", None) is None
        if isinstance(dx, NNDynamics):
            # networks the device dynamics do not cover (more than two hidden layers, wide
            # layers, other activations): torch runs the network (grad_input / autograd)
            try:
                dx._dilqr_pack(x_init.dtype, x_init.device)
            except NotImplementedError:
                generic_dx = True
        if not quad or generic_dx:
            # Module cost (approximate_cost, mpc.py:447-487) and / or a dynamics Module
            # without device kernels (AUTO_DIFF / FINITE_DIFF / ANALYTIC grad_input,
            # mpc.py:490-601): torch evaluates the Modules, the kernels run the sweeps
            return self._forward_generic(x_init, cost, dx, n_batch)
        C, c = self._expand_cost(cost, n_batch)
        if self.slew_rate_penalty is not None:
            return self._forward_slew(x_init, C, c, dx, n_batch)
        if isinstance(dx, NNDynamics):
            return self._forward_network(x_init, C, c, dx, n_batch)
        if isinstance(dx, LinDx):
            F, f = dx.F, dx.f
        else:
            F = f = None
        x, u, costs = self._Fn.apply(self, dx, x_init, C, c, F, f)
        return x, u, costs

    def _forward_slew(self, x_init, C, c, dx, n_batch):
        """Slew-rate penalty gamma * ||u_t - u_{t-1}||^2 by state augmentation
        x~ = (u_{t-1}, x) -- mpc.py:362-445.  The augmented problem is itself an LQR
        problem with linear dynamics, so it runs through the same kernels with
        n_state + n_ctrl states; autograd carries the KKT gradients of the augmented
        tensors back to C, c, F, f, x_init.  (The reference supports this only for
        Module dynamics -- its LinDx branch calls ``None`` at lqr_step.py:224 -- so the
        reference-equivalent entry is ``AffineDynamics``; LinDx is accepted as well.)"""
        if not isinstance(dx, LinDx):
            raise NotImplementedError("slew_rate_penalty: LinDx / AffineDynamics only")
        ns, nc, T = self.n_state, self.n_ctrl, self.T
        n, nt = ns + nc, ns + 2 * nc
        dt, dev = x_init.dtype, x_init.device
        F, f = dx.F, dx.f
        gamI = self.slew_rate_penalty * torch.eye(nc, dtype=dt, device=dev)
        _C = torch.zeros(T, n_batch, nt, nt, dtype=dt, device=dev)
        _C[:, :, :nc, :nc] = gamI
        _C[:, :, -nc:, :nc] = -gamI
        _C[:, :, :nc, -nc:] = -gamI
        _C[:, :, -nc:, -nc:] = gamI
        _C = _C + torch.nn.functional.pad(C, (nc, 0, nc, 0))
        _c = torch.cat((torch.zeros(T, n_batch, nc, dtype=dt, device=dev), c), 2)
        _F0 = torch.cat((torch.zeros(nc, n, dtype=dt, device=dev),
                         torch.eye(nc, dtype=dt, device=dev)), 1).expand(T - 1, n_batch, nc, nt)
        _F1 = torch.cat((torch.zeros(T - 1, n_batch, ns, nc, dtype=dt, device=dev), F), 3)
        _F = torch.cat((_F0, _F1), 2)
        _f = None
        if f is not None and f.nelement() > 0:
            _f = torch.cat((torch.zeros(T - 1, n_batch, nc, dtype=dt, device=dev), f), 2)
        if self.prev_ctrl is not None:
            prev_u = self.prev_ctrl.detach().to(device=dev, dtype=dt)
            while prev_u.ndimension() < 3:
                prev_u = prev_u.unsqueeze(0)
        else:
            prev_u = torch.zeros(1, n_batch, nc, dtype=dt, device=dev)
        _x_init = torch.cat((prev_u[0].expand(n_batch, nc), x_init), 1)
        inner = MPC(ns + nc, nc, T, u_lower=self.u_lower, u_upper=self.u_upper,
                    u_zero_I=self.u_zero_I, u_init=self.u_init, lqr_iter=self.lqr_iter,
                    grad_method=self.grad_method, verbose=self.verbose, eps=self.eps,
                    back_eps=self.back_eps, n_batch=n_batch,
                    linesearch_decay=self.linesearch_decay,
                    max_linesearch_iter=self.max_linesearch_iter,
                    exit_unconverged=self.exit_unconverged,
                    detach_unconverged=self.detach_unconverged, backprop=self.backprop,
                    not_improved_lim=self.not_improved_lim, best_cost_eps=self.best_cost_eps,
                    solo=self.solo, delta_u=self.delta_u)
        x, u, costs = inner(_x_init, QuadCost(_C, _c), LinDx(_F, _f))
        self.last_info = inner.last_info
        return x[:, :, nc:], u, costs

    # ------------------------------------------------------------------ generic Modules
    def approximate_cost(self, x, u, Cf, diff=True):
        """Second-order Taylor expansion of a cost Module along a trajectory (mpc.py:447-487):
        hessians [T,B,n,n], grads - H tau [T,B,n], costs [T,B].  All T timesteps go through
        the Module as one [T*B, n] batch (it acts row-wise), one autograd pass per column
        of the Hessian, on the device."""
        T, B = x.shape[0], x.shape[1]
        n = self.n_state + self.n_ctrl
        with torch.enable_grad():
            tau = torch.cat((x, u), 2).detach().reshape(T * B, n).requires_grad_()
            cost = Cf(tau)
            grad = torch.autograd.grad(cost.sum(), tau, create_graph=True, retain_graph=True)[0]
            cols = [torch.autograd.grad(grad[:, i].sum(), tau, retain_graph=True)[0] for i in range(n)]
            hess = torch.stack(cols, -1)
            grads = grad - torch.bmm(hess, tau.unsqueeze(2)).squeeze(2)
        out = (hess.reshape(T, B, n, n), grads.reshape(T, B, n), cost.reshape(T, B))
        return out if diff else tuple(t.detach() for t in out)

    def linearize_dynamics(self, x, u, dynamics, diff):
        """F[T-1,B,ns,n], f[T-1,B,ns] of a dynamics Module along (x, u) (mpc.py:490-601), all
        T-1 steps as one batch: ANALYTIC through ``dynamics.grad_input``, AUTO_DIFF through
        one autograd pass per state component, FINITE_DIFF by central differences
        (eps = 1e-4, util.py:10-20)."""
        T, B, ns, nc = self.T, x.shape[1], self.n_state, self.n_ctrl
        with torch.enable_grad():
            _x = x[:-1].reshape(-1, ns).detach().requires_grad_()
            _u = u[:-1].reshape(-1, nc).detach().requires_grad_()
            new_x = dynamics(_x, _u)
            if self.grad_method == GradMethods.ANALYTIC:
                if not diff:
                    R, S = dynamics.grad_input(_x.detach(), _u.detach())
                else:
                    R, S = dynamics.grad_input(_x, _u)
            elif self.grad_method == GradMethods.AUTO_DIFF:
                Rs, Ss = [], []
                for j in range(ns):
                    Rj, Sj = torch.autograd.grad(new_x[:, j].sum(), [_x, _u], retain_graph=True)
                    Rs.append(Rj)
                    Ss.append(Sj)
                R, S = torch.stack(Rs, 1), torch.stack(Ss, 1)
            elif self.grad_method == GradMethods.FINITE_DIFF:
                eps = 1e-4
                tau = torch.cat((_x, _u), 1).detach()
                cols = []
                for j in range(ns + nc):
                    e = torch.zeros(ns + nc, dtype=tau.dtype, device=tau.device)
                    e[j] = 1.
                    tp, tm = tau + eps * e, tau - eps * e
                    cols.append((dynamics(tp[:, :ns], tp[:, ns:]) - dynamics(tm[:, :ns], tm[:, ns:]))
                                / (2. * eps))
                J = torch.stack(cols, 2)
                if not diff:
                    J = J.detach()
                R, S = J[:, :, :ns], J[:, :, ns:]
            else:
                raise NotImplementedError("grad_method %s" % self.grad_method)
            if not diff:
                new_x, _x, _u = new_x.detach(), _x.detach(), _u.detach()
                R, S = R.detach(), S.detach()
            f = new_x - torch.bmm(R, _x.unsqueeze(2)).squeeze(2) - torch.bmm(S, _u.unsqueeze(2)).squeeze(2)
        F = torch.cat((R, S), 2).reshape(T - 1, B, ns, ns + nc)
        return F, f.reshape(T - 1, B, ns)

    def _forward_generic(self, x_init, cost, dx, n_batch):
        """MPC.forward for a cost Module and / or a dynamics Module without device kernels
        (mpc.py:248-337).  Per iLQR iteration torch evaluates and differentiates the
        Modules on the device (quadratic cost model, linearised dynamics, and the TRUE cost /
        dynamics inside the line search, lqr_step.py:164-261), batched over the problems and
        the horizon; the Riccati / pnqp sweep of every LQR step -- the hot part -- runs in
        the kernels on the resulting (C, c, F, f).  The gradient is the KKT adjoint at the
        solution with (C, c, F, f) re-derived under autograd (mpc.py:308-319)."""
        if self.slew_rate_penalty is not None:
            raise NotImplementedError("slew_rate_penalty with Module cost / dynamics: the reference "
                                      "itself exits here (mpc.py:451-457)")
        T, ns, nc = self.T, self.n_state, self.n_ctrl
        dt, dev = x_init.dtype, x_init.device
        quad = isinstance(cost, QuadCost)
        lin = isinstance(dx, LinDx)
        env = getattr(dx, "_dilqr_kind", None) is not None and not lin
        if quad:
            C, c = [t.detach().contiguous() for t in self._expand_cost(cost, n_batch)]

        def step(xt, ut, t):
            if lin:
                nx = torch.bmm(dx.F[t], torch.cat((xt, ut), 1).unsqueeze(2)).squeeze(2)
                return nx + dx.f[t] if (dx.f is not None and dx.f.nelement() > 0) else nx
            return dx(xt, ut).detach()

        def traj_cost(x, u):                                  # util.py:130-153
            tau = torch.cat((x, u), 2)
            if quad:
                return (0.5 * (torch.matmul(tau.unsqueeze(2), C) @ tau.unsqueeze(3)).reshape(T, -1)
                        + (tau * c).sum(2)).sum(0)
            return cost(tau.reshape(T * n_batch, ns + nc)).reshape(T, n_batch).sum(0)

        def bound(t, ut_nom):
            lo = self.u_lower if isinstance(self.u_lower, float) else self.u_lower[t]
            hi = self.u_upper if isinstance(self.u_upper, float) else self.u_upper[t]
            if self.delta_u is not None:                      # lqr_step.py:204-211
                lo = torch.maximum(ut_nom - self.delta_u, torch.as_tensor(lo, dtype=dt, device=dev))
                hi = torch.minimum(ut_nom + self.delta_u, torch.as_tensor(hi, dtype=dt, device=dev))
            return lo, hi

        if self.u_init is None:
            u = torch.zeros(T, n_batch, nc, dtype=dt, device=dev)
        else:
            u = self.u_init.detach().to(dt)
            if u.ndimension() == 2:
                u = u.unsqueeze(1).expand(T, n_batch, -1)
            u = u.clone()
        info = _solver.SolveInfo()
        eps_cmp = float(torch.tensor(self.eps, dtype=dt))
        best = None
        n_not_improved = 0
        with torch.no_grad():
            for i in range(self.lqr_iter):
                xs = [x_init.detach()]
                for t in range(T - 1):
                    xs.append(step(xs[t], u[t], t))
                x = torch.stack(xs, 0)
                if lin:
                    F, f = dx.F.detach(), (dx.f.detach() if dx.f is not None and dx.f.nelement() > 0 else None)
                elif env:
                    F, f = dx.linearize_traj(x, u)
                else:
                    F, f = self.linearize_dynamics(x, u, dx, diff=False)
                if not quad:
                    C, c, _ = self.approximate_cost(x, u, cost, diff=False)
                    C, c = C.contiguous(), c.contiguous()
                # lqr_backward (lqr_step.py:52-160) in the kernels: the gains of this LQR step
                _, _, _, li = _solver.solve_mpc(
                    x_init.detach(), C, c, _solver.DynSpec(_lib.DYN_LINDX, F=F, f=f), ns, nc, T,
                    u_lower=self.u_lower, u_upper=self.u_upper, u_zero_I=self.u_zero_I, u_init=u,
                    x_cur=x, lqr_iter=1, gain_solve=self._gain_solve, solo=self.solo, verbose=-1,
                    gains_only=True, delta_u=self.delta_u)
                K, k = li.K, li.k
                info.qp_iters.append(li.qp_iters[0] if li.qp_iters else 0)
                info.retries += li.retries
                # lqr_forward: line search on the TRUE cost / dynamics (lqr_step.py:164-261)
                old_cost = traj_cost(x, u)
                alphas = torch.ones(n_batch, dtype=dt, device=dev)
                cur, full_du, j = None, None, 0
                while (cur is None or bool((cur > old_cost).any())) and j < self.max_linesearch_iter:
                    nx, nu = [x_init.detach()], []
                    for t in range(T):
                        ut = torch.bmm(K[t], (nx[t] - x[t]).unsqueeze(2)).squeeze(2) + u[t] \
                            + alphas.unsqueeze(1) * k[t]
                        if self.u_zero_I is not None:
                            ut = ut.masked_fill(self.u_zero_I[t].to(torch.bool), 0.)
                        if self.u_lower is not None:
                            lo, hi = bound(t, u[t])
                            ut = torch.minimum(torch.maximum(ut, torch.as_tensor(lo, dtype=dt, device=dev)),
                                               torch.as_tensor(hi, dtype=dt, device=dev))
                        nu.append(ut)
                        if t < T - 1:
                            nx.append(step(nx[t], ut, t))
                    new_x, new_u = torch.stack(nx, 0), torch.stack(nu, 0)
                    cur = traj_cost(new_x, new_u)
                    if full_du is None:                       # lqr_step.py:243-245 (rows mix problems)
                        full_du = (u - new_u).transpose(1, 2).contiguous().view(n_batch, -1).norm(2, 1)
                    alphas = torch.where(cur > old_cost, alphas * self.linesearch_decay, alphas)
                    j += 1
                x, u, costs = new_x, new_u, cur
                n_not_improved += 1
                if best is None:                              # mpc.py:271-285
                    best = {"x": x.clone(), "u": u.clone(), "costs": costs.clone(), "du": full_du.clone()}
                else:
                    imp = costs <= best["costs"] + self.best_cost_eps
                    if bool(imp.any()):
                        n_not_improved = 0
                    best["x"][:, imp], best["u"][:, imp] = x[:, imp], u[:, imp]
                    best["costs"][imp], best["du"][imp] = costs[imp], full_du[imp]
                info.n_iters = i + 1
                if float(full_du.max()) < eps_cmp or n_not_improved > self.not_improved_lim:
                    break                                     # mpc.py:299-301
        x, u, costs = best["x"], best["u"], best["costs"]
        info.full_du_norm = best["du"]
        self.last_info = info
        mask = None
        if self.detach_unconverged and float(best["du"].max()) > eps_cmp:   # mpc.py:321-334
            if self.exit_unconverged:
                assert False
            if self.verbose >= 0:
                print("LQR Warning: All examples did not converge to a fixed point.")
                print("Detaching and *not* backpropping through the bad examples.")
            mask = (best["du"] < eps_cmp).to(dt)
        if not (self.backprop and torch.is_grad_enabled()):
            return x, u, costs
        # the final no-op LQR step under autograd (mpc.py:308-319)
        if lin:
            F = dx.F
            f = dx.f if (dx.f is not None and dx.f.nelement() > 0) else torch.zeros(
                T - 1, n_batch, ns, dtype=dt, device=dev)
        elif env:
            F, f = dx.linearize_traj(x, u)            # kernels: constants for autograd
        else:
            F, f = self.linearize_dynamics(x, u, dx, diff=True)
        if quad:
            Cg, cg = self._expand_cost(cost, n_batch)
        else:
            Cg, cg, _ = self.approximate_cost(x, u, cost, diff=True)
        xo, uo = _KKTAtSolutionFn.apply(self, mask, x_init, Cg.contiguous(), cg.contiguous(),
                                        F.contiguous(), f.contiguous(), x, u)
        return xo, uo, costs

    def _forward_network(self, x_init, C, c, dx, n_batch):
        """Module dynamics ``dynamics.NNDynamics`` (mpc.py:248-337 with
        grad_method=ANALYTIC): the iLQR solve runs in the kernels with the network as device
        dynamics -- the compiled ones for their shapes, the runtime-dimension ones for any
        other shape up to 32 variables (``_solver.nn_kernels``); the gradient is the KKT
        adjoint at the solution with F, f from ``linearize_dynamics(diff=True)``
        (mpc.py:490-523), a LinDx problem of the same shape."""
        if self.grad_method not in (GradMethods.ANALYTIC, GradMethods.AUTO_DIFF,
                                    GradMethods.FINITE_DIFF):
            raise NotImplementedError("Module dynamics: grad_method %s" % self.grad_method)
        # AUTO_DIFF (mpc.py:541-551) differentiates the same network: it is served by the
        # analytic grad_input Jacobian.  FINITE_DIFF (mpc.py:567-583): central differences
        # of the step, eps = 1e-4, in the kernel and (with autograd) at the solution.
        fd = self.grad_method == GradMethods.FINITE_DIFF
        dt, dev = x_init.dtype, x_init.device
        aux, ints = dx._dilqr_pack(dt, dev)
        ints[3] = 1 if fd else 0
        dyn = _solver.DynSpec(_lib.DYN_NN, aux=aux, ai=ints)
        x, u, costs, info = _solver.solve_mpc(
            x_init, C, c, dyn, self.n_state, self.n_ctrl, self.T,
            u_lower=self.u_lower, u_upper=self.u_upper, u_zero_I=self.u_zero_I,
            u_init=self.u_init, lqr_iter=self.lqr_iter, eps=self.eps,
            linesearch_decay=self.linesearch_decay,
            max_linesearch_iter=self.max_linesearch_iter,
            not_improved_lim=self.not_improved_lim, best_cost_eps=self.best_cost_eps,
            gain_solve=self._gain_solve, solo=self.solo, verbose=self.verbose,
            delta_u=self.delta_u)
        self.last_info = info
        mask = None
        eps_cmp = float(torch.tensor(self.eps, dtype=dt))
        if self.detach_unconverged:                      # mpc.py:321-334
            if float(info.full_du_norm.max()) > eps_cmp:
                if self.exit_unconverged:
                    assert False
                if self.verbose >= 0:
                    print("LQR Warning: All examples did not converge to a fixed point.")
                    print("Detaching and *not* backpropping through the bad examples.")
                mask = (info.full_du_norm < eps_cmp).to(dt)
        if not (self.backprop and torch.is_grad_enabled()):
            return x, u, costs
        # linearise at the solution WITH the autograd graph (mpc.py:496-523)
        T, ns, nc = self.T, self.n_state, self.n_ctrl
        _x = x[:-1].reshape(-1, ns)
        _u = u[:-1].reshape(-1, nc)
        if fd:                                           # util.py:10-20, batched
            eps = 1e-4
            tau = torch.cat((_x, _u), 1)
            cols = []
            for j in range(ns + nc):
                e = torch.zeros(ns + nc, dtype=dt, device=dev)
                e[j] = 1.
                tp, tm = tau + eps * e, tau - eps * e
                cols.append((dx(tp[:, :ns], tp[:, ns:]) - dx(tm[:, :ns], tm[:, ns:])) / (2. * eps))
            J = torch.stack(cols, 2)
            R, S = J[:, :, :ns], J[:, :, ns:]
            new_x = dx(_x, _u)
        else:
            new_x = dx(_x, _u)
            R, S = dx.grad_input(_x, _u)
            if self.grad_method == GradMethods.AUTO_DIFF:
                # the reference takes these Jacobians with torch.autograd.grad WITHOUT
                # create_graph (mpc.py:544-551): they are constants for the backward pass,
                # the network's parameters are reached through f only
                R, S = R.detach(), S.detach()
        f = new_x - torch.bmm(R, _x.unsqueeze(2)).squeeze(2) - torch.bmm(S, _u.unsqueeze(2)).squeeze(2)
        F = torch.cat((R, S), 2).reshape(T - 1, n_batch, ns, ns + nc)
        f = f.reshape(T - 1, n_batch, ns)
        Cd = C if C.is_contiguous() else C.contiguous()
        cd = c if c.is_contiguous() else c.contiguous()
        xo, uo = _KKTAtSolutionFn.apply(self, mask, x_init, Cd, cd, F, f, x, u)
        return xo, uo, costs
