"""``mpc_explicit.MPC`` -- drop-in for the reference's DiLQR variant
(mpc_explicit.py:58-358 + lqr_step_explicit.py): same forward as ``mpc.MPC``
with the analytic env_dx linearisation (mpc_explicit.py:516-546), and the
implicit fixed-point gradient wrt the cost (C, c) and the dynamics parameters
``dx.params`` in the backward pass (lqr_step_explicit.py:652-712)."""
import torch
from torch.autograd import Function

from . import _lib, _solver
from .definitions import QuadCost, LinDx  # noqa: F401
from .mpc import MPC as _BaseMPC, GradMethods, _dyn_spec  # noqa: F401


class _MPCExplicitFn(Function):
    """``q, p``: set when (C, c) is the tiled diagonal cost of il_env.py:159-162 built by
    ``il.tile_cost`` -- C, c then come in detached and the backward returns the gradient wrt
    (q, p) directly (the adjoint of the tiling is accumulated inside the final adjoint pass;
    the dense dC[T,B,n,n] is never written)."""

    @staticmethod
    def forward(ctx, mod, dx, x_init, C, c, theta, q=None, p=None):
        ctx.set_materialize_grads(False)
        ctx.tiled = q is not None
        deferred = mod.deferred if (mod.defer_checks and not (
            mod.detach_unconverged and (mod.exit_unconverged or mod.verbose >= 0))) else None
        dyn = _dyn_spec(dx)
        # A 4-D stride-0 cost (e.g. Q[None, None].expand(T, B, n, n)) is read as the broadcast
        # block it is -- unless its gradient is wanted: autograd then expects a [T,B,n,n]
        # gradient per (t, b) like the reference returns, so the dense tensor is used.
        if C.ndimension() == 4 and ctx.needs_input_grad[3]:
            C = C.contiguous()
        if c.ndimension() == 3 and ctx.needs_input_grad[4]:
            c = c.contiguous()
        x, u, costs, info = _solver.solve_mpc(
            x_init, C, c, dyn, mod.n_state, mod.n_ctrl, mod.T,
            u_lower=mod.u_lower, u_upper=mod.u_upper, u_zero_I=mod.u_zero_I,
            u_init=mod.u_init, lqr_iter=mod.lqr_iter, eps=mod.eps,
            linesearch_decay=mod.linesearch_decay,
            max_linesearch_iter=mod.max_linesearch_iter,
            not_improved_lim=mod.not_improved_lim, best_cost_eps=mod.best_cost_eps,
            gain_solve=_lib.GAIN_PLAIN, solo=mod.solo, verbose=mod.verbose, delta_u=mod.delta_u,
            deferred=deferred)
        mod.last_info = info
        ctx.mod, ctx.dx = mod, dx
        ctx.deferred = deferred
        ctx.theta_host = dyn.params
        ctx.mask = None
        eps_cmp = float(torch.tensor(mod.eps, dtype=x.dtype))
        if mod.detach_unconverged:                       # mpc_explicit.py:343-356
            # the mask is a device op; only the reference's warning / assert needs the host
            # to look at the norms (one sync), so a quiet caller (verbose < 0) pays none
            mask = (info.full_du_norm < eps_cmp).to(x.dtype)
            if mod.exit_unconverged or mod.verbose >= 0:
                if float(info.full_du_norm.max()) > eps_cmp:
                    if mod.exit_unconverged:
                        assert False
                    print("LQR Warning: All examples did not converge to a fixed point.")
                    print("Detaching and *not* backpropping through the bad examples.")
                else:
                    mask = None
            ctx.mask = mask
        ctx.save_for_backward(x_init, C, c, x, u)
        ctx.mark_non_differentiable(costs)
        # a gradient wrt the cost or theta will be asked for: enqueue the part of the
        # backward that only needs the solution right behind the solve (the final no-op
        # LQR pass is part of the reference's forward too, mpc_explicit.py:325-340)
        ctx.prep = None
        if mod.backprop and mod.prepare_in_forward and any(ctx.needs_input_grad[3:8]):
            ctx.prep = _solver.dilqr_prepare(
                x_init, C, c, x, u, dx, mod.n_state, mod.n_ctrl, mod.u_lower, mod.u_upper,
                solo=mod.solo, theta_host=dyn.params, solve_info=info, deferred=deferred)
        return x, u, costs

    @staticmethod
    def backward(ctx, dl_dx, dl_du, _dcosts):
        mod, dx = ctx.mod, ctx.dx
        x_init, C, c, x, u = ctx.saved_tensors
        if ctx.mask is not None:
            dl_dx = None if dl_dx is None else dl_dx * ctx.mask.view(1, -1, 1)
            dl_du = None if dl_du is None else dl_du * ctx.mask.view(1, -1, 1)
        stats = {}
        dC, dc, dtheta = _solver.dilqr_backward(
            dl_dx, dl_du, x_init, C, c, x, u, dx, mod.n_state,
            mod.n_ctrl, mod.u_lower, mod.u_upper, n_passes=mod.richardson_passes,
            tol=mod.richardson_tol, back_eps=mod.back_eps, solo=mod.solo, stats=stats,
            theta_host=ctx.theta_host, prep=ctx.prep, tile_reduce=ctx.tiled,
            deferred=ctx.deferred, solver=mod.adjoint_solver, gmres_restart=mod.gmres_restart,
            gmres_tol=mod.gmres_tol, gmres_max_iter=mod.gmres_max_iter)
        ctx.prep = None
        mod.last_backward = stats
        # dC / dc come back in the layout of the cost tensors handed in (dense, or already
        # summed over the broadcast axes for C[n,n] / C[T,n,n]); the reference returns
        # dtheta[B, n_theta] and autograd sums it to theta's shape
        dth = None
        if ctx.needs_input_grad[5]:      # dx.params may live on the host (PendulumDx() default)
            dth = dtheta.sum(0).to(device=dx.params.device, dtype=dx.params.dtype)
        if ctx.tiled:                    # (dC, dc) are already (dq, dp)
            return None, None, None, None, None, dth, dC, dc
        return None, None, None, dC.reshape(C.shape), dc.reshape(c.shape), dth, None, None


class MPC(_BaseMPC):
    """Arguments as the reference (mpc_explicit.py:122-143) plus the solver of the
    matrix-free fixed-point system A'w = g of the backward:

    - ``adjoint_solver="richardson"`` (default): ``richardson_passes`` (max adjoint-LQR
      passes) and ``richardson_tol`` (relative stop tolerance; None = fixed pass count).
      Converges only where the iteration matrix M = I - A has rho(M) < 1 (a converged
      iLQR fixed point).
    - ``adjoint_solver="gmres"``: restarted GMRES per problem, the reference's dense solve
      wherever A is nonsingular; ``gmres_restart`` basis vectors per cycle (clipped to T n),
      ``gmres_tol`` relative residual (None: 1e-12 in FP64, 1e-5 in FP32), ``gmres_max_iter``
      Arnoldi steps (None: 2 T n).  See ``_solver.dilqr_backward``."""

    def __init__(self, *args, richardson_passes=30, richardson_tol=1e-14,
                 prepare_in_forward=True, adjoint_solver="richardson", gmres_restart=64,
                 gmres_tol=None, gmres_max_iter=None, **kw):
        super().__init__(*args, **kw)
        self.prepare_in_forward = prepare_in_forward
        # defer_checks: postpone every validation read of a step (pnqp trace, stop-rule
        # status, adjoint line-search test) to ONE host sync when the caller resolves
        # `self.deferred` (il.ImitationStep does); a failed check means "repeat the step
        # with immediate checks".  Off by default: MPC.forward then returns validated data.
        self.defer_checks = False
        self.deferred = None
        self.richardson_passes = richardson_passes
        self.richardson_tol = richardson_tol
        if adjoint_solver not in ("richardson", "gmres"):
            raise ValueError("adjoint_solver must be 'richardson' or 'gmres', got %r"
                             % (adjoint_solver,))
        self.adjoint_solver = adjoint_solver
        self.gmres_restart = gmres_restart
        self.gmres_tol = gmres_tol
        self.gmres_max_iter = gmres_max_iter
        self.last_backward = None

    def forward(self, x_init, cost, dx):
        if isinstance(dx, LinDx):
            # the reference's explicit variant rejects LinDx (mpc_explicit.py:325)
            raise AttributeError("'LinDx' object has no attribute 'params'")
        if not isinstance(cost, QuadCost):
            raise NotImplementedError("only QuadCost is supported (SURVEY 8a-2)")
        if self.slew_rate_penalty is not None:
            raise NotImplementedError("slew_rate_penalty: supported by mpc.MPC (LinDx / "
                                      "AffineDynamics); the env_dx models have no "
                                      "control-passthrough kernels")
        n_batch = self.n_batch if self.n_batch is not None else (
            cost.C.size(1) if cost.C.ndimension() == 4 else None)
        if n_batch is None:
            print('MPC Error: Could not infer batch size, pass in as n_batch')
            import sys
            sys.exit(-1)
        self._expand_cost(cost, n_batch)      # shape validation (mpc_explicit.py:203-224)
        assert x_init.ndimension() == 2 and x_init.size(0) == n_batch
        # broadcast costs (C[n,n], C[T,n,n]) are NOT tiled: the kernels read the shared
        # block and the backward returns the gradient already reduced to that shape
        tile = getattr(cost.C, "_dilqr_tile", None)
        if tile is not None and getattr(cost.c, "_dilqr_tile", None) is tile:
            q, p = tile
            return _MPCExplicitFn.apply(self, dx, x_init, cost.C.detach(), cost.c.detach(),
                                        dx.params, q, p)
        return _MPCExplicitFn.apply(self, dx, x_init, cost.C, cost.c, dx.params)
