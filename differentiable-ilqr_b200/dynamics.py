"""Dynamics containers of the upstream mpc.pytorch API kept by the reference
(dynamics.py): ``NNDynamics``, ``AffineDynamics`` and ``CtrlPassthroughDynamics``.

``NNDynamics`` with one or two hidden layers (sigmoid or relu; at most 128 units in the first
of two layers) runs inside the iteration kernels as device dynamics, for any shape with
``n_state + n_ctrl <= 32``: ``DILQR_DYN_NN`` (csrc/dynamics.cuh) on the compiled shapes,
``DILQR_DYN_NN_RT`` (csrc/rt_kernels.cuh) on every other one.  ``MPC.forward`` packs the weights
once per call; the KKT gradients ``dF, df`` of the solve reach the weights through
``grad_input`` evaluated (with autograd) at the solution, which is what the reference
does in ``linearize_dynamics(diff=True)`` (mpc.py:490-523).

``AffineDynamics`` is a time-invariant LinDx: ``MPC.forward`` hands the solver
``F = [A B]`` and ``f = c`` broadcast over (T-1, B) and autograd sums the KKT
gradients ``dF, df`` back to ``A, B, c`` -- which is what the reference computes
through ``linearize_dynamics(diff=True)`` (mpc.py:504-523: ``f = x' - R x - S u``
is identically ``c``).  ``forward`` / ``grad_input`` are plain tensor expressions
for callers that simulate the plant; the solve itself never calls them.
"""
import torch
from torch import nn


ACTS = {'sigmoid': torch.sigmoid, 'relu': torch.relu, 'elu': torch.nn.functional.elu}


class NNDynamics(nn.Module):
    """dynamics.py:15-130: fully connected network x' = net([x, u]) (+ x)."""

    def __init__(self, n_state, n_ctrl, hidden_sizes=[100], activation='sigmoid',
                 passthrough=True):
        super().__init__()
        assert activation in ACTS
        self.passthrough = passthrough
        self.activation = activation
        sizes = [n_state + n_ctrl] + list(hidden_sizes) + [n_state]
        self.fcs = nn.ModuleList(nn.Linear(a, b) for a, b in zip(sizes[:-1], sizes[1:]))
        self.zs = []      # hidden activations of the last forward (used by grad_input)

    @property
    def Ws(self):
        return [fc.weight for fc in self.fcs]

    def forward(self, x, u):                               # dynamics.py:57-79
        x_dim = x.ndimension()
        if x_dim == 1:
            x = x.unsqueeze(0)
        if u.ndimension() == 1:
            u = u.unsqueeze(0)
        z = torch.cat((x, u), 1)
        zs = []
        for i, fc in enumerate(self.fcs):
            z = fc(z)
            if i < len(self.fcs) - 1:
                z = ACTS[self.activation](z)
                zs.append(z)
        self.zs = zs
        if self.passthrough:
            z = z + x
        return z.squeeze(0) if x_dim == 1 else z

    def grad_input(self, x, u):                            # dynamics.py:81-130
        """R = dx'/dx, S = dx'/du at the inputs of the LAST forward call."""
        x_dim = x.ndimension()
        n_batch, n_state = x.shape[-2] if x_dim > 1 else 1, x.shape[-1]
        diff = x.requires_grad or u.requires_grad or torch.is_grad_enabled()
        Ws = self.Ws if diff else [W.detach() for W in self.Ws]
        zs = self.zs if diff else [z.detach() for z in self.zs]
        assert len(zs) == len(Ws) - 1
        grad = Ws[-1].unsqueeze(0).expand(n_batch, -1, -1)
        for i in range(len(zs) - 1, -1, -1):
            if self.activation == 'relu':
                d = (zs[i] > 0.).to(zs[i].dtype)
            elif self.activation == 'sigmoid':
                d = zs[i] * (1. - zs[i])
            else:
                assert False
            grad = grad.bmm(Ws[i].unsqueeze(0) * d.unsqueeze(2))
        R, S = grad[:, :, :n_state], grad[:, :, n_state:]
        if self.passthrough:
            R = R + torch.eye(n_state, dtype=R.dtype, device=R.device).unsqueeze(0)
        if x_dim == 1:
            R, S = R.squeeze(0), S.squeeze(0)
        return R, S

    # -- device side ---------------------------------------------------------
    def _dilqr_pack(self, dtype, device):
        """(weight buffer, ints) for DILQR_DYN_NN / DILQR_DYN_NN_RT: weight[out][in], bias[out]
        per layer."""
        if len(self.fcs) not in (2, 3):
            raise NotImplementedError("device NNDynamics: one or two hidden layers; got %d"
                                      % (len(self.fcs) - 1))
        widths = [fc.weight.shape[0] for fc in self.fcs[:-1]]
        if max(widths) >= 65536 or (len(widths) == 2 and widths[0] > 128):
            raise NotImplementedError("device NNDynamics: hidden widths %s too large" % widths)
        if self.activation not in ('sigmoid', 'relu'):
            raise NotImplementedError("device NNDynamics: sigmoid / relu (grad_input of the "
                                      "reference supports no other, dynamics.py:104-113)")
        buf = torch.cat([t.detach().reshape(-1) for fc in self.fcs
                         for t in (fc.weight, fc.bias)]).to(device=device, dtype=dtype)
        ints = [widths[0] | ((widths[1] << 16) if len(widths) == 2 else 0),
                0 if self.activation == 'sigmoid' else 1, 1 if self.passthrough else 0, 0]
        return buf.contiguous(), ints


class AffineDynamics(nn.Module):
    def __init__(self, A, B, c=None):
        super().__init__()
        assert A.ndimension() == 2
        assert B.ndimension() == 2
        if c is not None:
            assert c.ndimension() == 1
        self.A, self.B, self.c = A, B, c

    def forward(self, x, u):                               # dynamics.py:173-195
        x_dim = x.ndimension()
        if x_dim == 1:
            x = x.unsqueeze(0)
        if u.ndimension() == 1:
            u = u.unsqueeze(0)
        z = x.mm(self.A.t()) + u.mm(self.B.t())
        if self.c is not None:
            z = z + self.c
        return z.squeeze(0) if x_dim == 1 else z

    def grad_input(self, x, u):                            # dynamics.py:197-202
        n_batch = x.size(0)
        return (self.A.unsqueeze(0).repeat(n_batch, 1, 1),
                self.B.unsqueeze(0).repeat(n_batch, 1, 1))

    def as_lindx(self, T, n_batch, dtype, device):
        """F[T-1,B,ns,ns+nc], f[T-1,B,ns] (or None) as differentiable views."""
        ns = self.A.shape[0]
        Fm = torch.cat((self.A, self.B), 1).to(device=device, dtype=dtype)
        F = Fm.unsqueeze(0).unsqueeze(0).expand(T - 1, n_batch, ns, Fm.shape[1])
        f = None
        if self.c is not None:
            f = self.c.to(device=device, dtype=dtype).unsqueeze(0).unsqueeze(0).expand(
                T - 1, n_batch, ns)
        return F, f


class CtrlPassthroughDynamics(nn.Module):
    """x~ = (u_prev, x): the augmented plant of the slew-rate formulation
    (dynamics.py:133-156)."""

    def __init__(self, dynamics):
        super().__init__()
        self.dynamics = dynamics

    def forward(self, tilde_x, u):
        dim = tilde_x.ndimension()
        if dim == 1:
            tilde_x = tilde_x.unsqueeze(0)
        if u.ndimension() == 1:
            u = u.unsqueeze(0)
        n_ctrl = u.size(1)
        xtp1 = self.dynamics(tilde_x[:, n_ctrl:], u)
        out = torch.cat((u, xtp1), dim=1)
        return out.squeeze() if dim == 1 else out

    def grad_input(self, x, u):
        assert False, "Unimplemented"                      # dynamics.py:155-156
