"""Imitation-learning step in the shape of the reference's ``il_exp`` loop
(il_exp.py:326-409) and ``IL_Env.mpc`` (il_env.py:153-188): tile the diagonal
cost, solve the batched MPC, imitation loss against expert controls, implicit
backward to (theta, q, p).  Problems are sharded across ranks by batch index;
the only collective is one all-reduce of the (n_theta + 2 n) gradient scalars.
"""
import torch

import ctypes as C

from torch.autograd import Function

from . import _lib, mpc_explicit, parallel
from ._solver import _DT, _ptr, _stream, Deferred
from .definitions import QuadCost


class TileCost(Function):
    """(q[n], p[n]) -> dense C[T,B,n,n] = diag(q), c[T,B,n] = p, the tensors
    il_env.py:159-162 builds with ``.repeat``; the backward is the adjoint of that
    tiling (what autograd does for the reference at il_exp.py:373) as one streaming
    reduction kernel instead of a strided torch sum."""

    @staticmethod
    def forward(ctx, q, p, T, B):
        n = q.shape[0]
        q_, p_ = q.detach().contiguous(), p.detach().contiguous()
        Cm = torch.empty(T, B, n, n, dtype=q.dtype, device=q.device)
        cv = torch.empty(T, B, n, dtype=q.dtype, device=q.device)
        _lib.call("dilqr_tile_cost", _DT[q.dtype], n, T, B, _ptr(q_), _ptr(p_), _ptr(Cm), _ptr(cv),
                  _stream())
        ctx.dims = (n, T, B)
        return Cm, cv

    @staticmethod
    def backward(ctx, dC, dc):
        n, T, B = ctx.dims
        if dC is None:
            dC = torch.zeros(T, B, n, n, dtype=dc.dtype, device=dc.device)
        if dc is None:
            dc = torch.zeros(T, B, n, dtype=dC.dtype, device=dC.device)
        dC, dc = dC.contiguous(), dc.contiguous()
        dq = torch.empty(n, dtype=dC.dtype, device=dC.device)
        dp = torch.empty(n, dtype=dC.dtype, device=dC.device)
        nbytes = _lib.lib().dilqr_tile_cost_grad_workspace_bytes(n)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dC.device)
        _lib.call("dilqr_tile_cost_grad", _DT[dC.dtype], n, T, B, _ptr(dC), _ptr(dc), _ptr(dq),
                  _ptr(dp), _ptr(ws), C.c_size_t(nbytes), _stream())
        return dq, dp, None, None


def tile_cost(q, p, T, B):
    """il_env.py:159-162 as one call: (C[T,B,n,n] = diag(q), c[T,B,n] = p).  The pair is
    tagged with its source so that ``mpc_explicit.MPC`` can hand the gradient wrt (q, p)
    back directly -- the adjoint of the tiling is then accumulated inside the final adjoint
    pass and the dense dC (0.94 GB at T=50, B=65536) is neither written nor re-read.
    Used on their own (any other consumer), C and c are ordinary autograd tensors."""
    Cm, cv = TileCost.apply(q, p, T, B)
    tag = (q, p)
    Cm._dilqr_tile = tag
    cv._dilqr_tile = tag
    return Cm, cv


class ImitationStep:
    def __init__(self, dx_cls, T, lqr_iter, dtype, device, n_richardson=4, richardson_tol=None,
                 group=None, tile=True, detach_unconverged=False, adjoint_solver="richardson",
                 gmres_restart=64, gmres_tol=None, gmres_max_iter=None):
        # adjoint_solver / gmres_*: the solver of the backward's adjoint system, as in
        # mpc_explicit.MPC (the GMRES status is read in the step's one deferred host sync)
        # tile=True: materialise Q,p as [T,B,n,n] / [T,B,n] exactly like il_env.py:159-162;
        # tile=False: hand MPC the [n,n] / [n] tensors (mpc.py:205-219 broadcasts them)
        self.tile = tile
        self.dx_cls = dx_cls
        self.T = T
        self.dtype, self.device = dtype, device
        proto = dx_cls()
        self.ns, self.nc = proto.n_state, proto.n_ctrl
        self.mpc = mpc_explicit.MPC(
            self.ns, self.nc, T, u_lower=proto.lower, u_upper=proto.upper, lqr_iter=lqr_iter,
            verbose=-1, exit_unconverged=False, detach_unconverged=detach_unconverged,
            linesearch_decay=proto.linesearch_decay,
            max_linesearch_iter=proto.max_linesearch_iter, eps=proto.mpc_eps,
            richardson_passes=n_richardson, richardson_tol=richardson_tol,
            adjoint_solver=adjoint_solver, gmres_restart=gmres_restart, gmres_tol=gmres_tol,
            gmres_max_iter=gmres_max_iter)
        self.group = group
        self.retries = 0
        self.redone = 0           # steps repeated because a deferred check failed
        self.backward_name = ("DiLQR implicit (%d Richardson passes)" % n_richardson
                              if adjoint_solver == "richardson" else
                              "DiLQR implicit (GMRES(%d))" % gmres_restart)
        self.d2h_bytes = 0
        self.defer = True         # one host sync per step (see _solver.Deferred)
        self._out_host = None
        self._h2d = None          # side stream of run_host
        self._uexp_ready = None

    # -- pieces -----------------------------------------------------------
    def tile_cost(self, q, p, B):
        """il_env.py:159-162: Q = diag(q) tiled to [T,B,n,n], p tiled to [T,B,n]."""
        if not self.tile:
            return torch.diag(q), p
        return tile_cost(q, p, self.T, B)

    def prepare(self, x0, q, p, theta):
        return {"x0": x0, "q": q.clone().requires_grad_(), "p": p.clone().requires_grad_(),
                "theta": theta.clone().requires_grad_(),
                "theta_host": theta.detach().double().cpu().tolist()}

    def _step(self, x0, uexp, q, p, theta, world_frac=1.0, theta_host=None, defer=None):
        """One il_exp step.  Nothing in it waits for the device: the kernels take theta
        by value from ``theta_host`` (the caller's host copy; without it the parameters are
        read back once, before anything is queued) and every validation read is deferred to
        the end of the step (``_solver.Deferred``), where the caller synchronises anyway to
        fetch the loss.  Returns (flat, deferred)."""
        defer = self.defer if defer is None else defer
        for t in (q, p, theta):
            t.grad = None
        B = x0.shape[0]
        self.mpc.n_batch = B
        dx = self.dx_cls(theta)
        if theta_host is not None:
            dx.set_host_params(theta_host)
        else:
            dx._theta_list()      # the one device->host read of a step, before anything is queued
        self.mpc.defer_checks = defer
        self.mpc.deferred = Deferred() if defer else None
        C, c = self.tile_cost(q, p, B)
        x, u, _ = self.mpc(x0, QuadCost(C, c), dx)
        if self._uexp_ready is not None:   # run_host: uexp was copied on a side stream
            torch.cuda.current_stream().wait_event(self._uexp_ready)
        # loss = mean((u - u_expert)^2) (il_exp.py:346) and loss.backward() (il_exp.py:373) with
        # the gradient of the loss written out by hand: d loss / du = 2 (u - u_expert) / numel.
        # Three small kernels instead of the dozen of the pow / mean / mul autograd chain -- at
        # this point of the step the device is waiting for the host.
        with torch.no_grad():
            d = u - uexp
            scale = world_frac / d.numel()
            loss = torch.dot(d.reshape(-1), d.reshape(-1)) * scale
            gu = d * (2.0 * scale)
        torch.autograd.backward([u], [gu])
        flat = torch.cat((theta.grad, q.grad, p.grad, loss.reshape(1)))
        return parallel.allreduce_sum_(flat, self.group), self.mpc.deferred

    def _checked(self, run):
        """Run a step optimistically; if one of its deferred checks fails (a pnqp trace
        guess was wrong, or an adjoint step would have been rejected) repeat it with
        immediate checks -- still entirely on the device."""
        flat, d = run(None)
        if d is not None and not d.resolve():
            self.redone += 1
            flat, _ = run(False)
        self.retries += self.mpc.last_info.retries
        return flat

    # -- resident inputs (device timing) -----------------------------------
    def run_resident(self, res, uexp):
        w = 1.0
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            w = 1.0 / torch.distributed.get_world_size()
        return self._checked(lambda defer: self._step(
            res["x0"], uexp, res["q"], res["p"], res["theta"], w, res.get("theta_host"), defer))

    # -- host inputs (end to end) -------------------------------------------
    def run_host(self, x0_h, uexp_h, q_h, p_h, theta_h):
        dev = self.device
        main = torch.cuda.current_stream(dev)
        x0 = x0_h.to(dev, non_blocking=True)
        # the expert controls (the bulk of the inputs: T*B*nc scalars) are first needed by the
        # loss, after the solve: their copy runs on a side stream next to the solve instead of
        # in front of it.  The side stream starts behind everything already queued on the
        # caller's stream, so the copy stays inside the step.
        if self._h2d is None:
            self._h2d = torch.cuda.Stream(dev)
        self._h2d.wait_stream(main)
        with torch.cuda.stream(self._h2d):
            uexp = uexp_h.to(dev, non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(self._h2d)
        uexp.record_stream(main)
        self._uexp_ready = ready
        q = q_h.to(dev, non_blocking=True).requires_grad_()
        p = p_h.to(dev, non_blocking=True).requires_grad_()
        theta = theta_h.to(dev, non_blocking=True).requires_grad_()
        w = 1.0
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            w = 1.0 / torch.distributed.get_world_size()
        th_host = theta_h.double().tolist()
        out = None

        def run(defer):
            nonlocal out
            flat, d = self._step(x0, uexp, q, p, theta, w, th_host, defer)
            # loss + gradients back to the host: enqueued behind the step, ONE sync serves
            # this copy and the deferred checks
            if self._out_host is None or self._out_host.numel() != flat.numel():
                self._out_host = torch.empty(flat.numel(), dtype=flat.dtype).pin_memory()
            self._out_host.copy_(flat, non_blocking=True)
            return flat, d

        self._checked(run)
        self._uexp_ready = None
        torch.cuda.current_stream().synchronize()
        out = self._out_host.clone()
        self.d2h_bytes = out.numel() * out.element_size()
        return out


class ImitationLearner:
    """The `il_exp --mode empc` loop (il_exp.py:183-429) on the device: learn the dynamics
    parameters theta (`learn_dx`) and / or the cost (`learn_cost`: q = sigmoid(q_logit),
    p = sqrt(q) * learn_p, il_exp.py:127-133,331-333) by differentiating the imitation loss
    mean((u_mpc - u_expert)^2) through the MPC (DiLQR implicit gradient), RMSprop lr 1e-2
    alpha 0.5 (il_exp.py:228-238), warm-start cache of the previous controls
    (il_exp.py:269-275,338-344).  Under torch.distributed each rank owns a contiguous
    shard of the problems (parallel.shard_range) and one small all-reduce per step sums
    the parameter gradients; every rank then takes the identical optimiser step."""

    def __init__(self, dx_cls, theta_init, T, lqr_iter=100, dtype=torch.float64,
                 device=None, lr=1e-2, alpha=0.5, richardson_passes=30, richardson_tol=1e-10,
                 group=None, learn_dx=True, learn_cost=False, adjoint_solver="richardson",
                 gmres_restart=64, gmres_tol=None, gmres_max_iter=None):
        self.dx_cls, self.T = dx_cls, T
        self.dtype, self.device, self.group = dtype, device, group
        self.learn_dx, self.learn_cost = learn_dx, learn_cost
        proto = dx_cls()
        self.ns, self.nc = proto.n_state, proto.n_ctrl
        self.q, self.p = [t.to(dtype).to(device) for t in proto.get_true_obj()]
        self.theta = torch.tensor(theta_init, dtype=dtype, device=device, requires_grad=learn_dx)
        # il_exp.py:127-133: the learnt cost starts from q = 1/2, p = 0
        self.learn_q_logit = torch.zeros_like(self.q, requires_grad=learn_cost)
        self.learn_p = torch.zeros_like(self.p, requires_grad=learn_cost)
        self.params = ([self.learn_q_logit, self.learn_p] if learn_cost else []) + (
            [self.theta] if learn_dx else [])
        self.opt = torch.optim.RMSprop([{"params": self.params, "lr": lr, "alpha": alpha}])
        self.mpc = mpc_explicit.MPC(
            self.ns, self.nc, T, u_lower=proto.lower, u_upper=proto.upper, lqr_iter=lqr_iter,
            verbose=-1, exit_unconverged=False, detach_unconverged=True,
            linesearch_decay=proto.linesearch_decay,
            max_linesearch_iter=proto.max_linesearch_iter, eps=proto.mpc_eps,
            richardson_passes=richardson_passes, richardson_tol=richardson_tol,
            adjoint_solver=adjoint_solver, gmres_restart=gmres_restart, gmres_tol=gmres_tol,
            gmres_max_iter=gmres_max_iter)
        self.warm = None

    def cost(self):
        """(q, p) the controller runs with (il_exp.py:331-335)."""
        if self.learn_cost:
            q = torch.sigmoid(self.learn_q_logit)
            return q, q.sqrt() * self.learn_p
        return self.q, self.p

    def expert(self, theta_true, x_init):
        """populate_data (il_env.py:81-94): one batched open-loop solve with the true model."""
        dx = self.dx_cls(torch.tensor(theta_true, dtype=self.dtype, device=self.device))
        self.mpc.n_batch = x_init.shape[0]
        self.mpc.u_init = None
        with torch.no_grad():
            _, u, _ = self.mpc(x_init, QuadCost(torch.diag(self.q), self.p), dx)
        return u

    def step(self, x_init, u_expert, n_global=None):
        """One il_exp training step on this rank's shard; returns the global loss."""
        B = x_init.shape[0]
        n_global = n_global or B
        self.opt.zero_grad()
        self.mpc.n_batch = B
        self.mpc.u_init = self.warm
        dx = self.dx_cls(self.theta)
        q, p = self.cost()
        _, u, _ = self.mpc(x_init, QuadCost(torch.diag(q), p), dx)
        self.warm = u.detach()
        # mean over the GLOBAL batch: local sum / (T * n_global * nc)
        loss = (u - u_expert).pow(2).sum() / (self.T * n_global * self.nc)
        loss.backward()
        flat = torch.cat([t.grad.reshape(-1) for t in self.params] + [loss.detach().reshape(1)])
        parallel.allreduce_sum_(flat, self.group)
        off = 0
        for t in self.params:
            t.grad.copy_(flat[off:off + t.numel()].view_as(t))
            off += t.numel()
        self.opt.step()
        return float(flat[-1])
