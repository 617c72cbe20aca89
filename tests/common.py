"""Helpers shared by the tests (problem generators, golden loader, the kernel-family table)."""
import importlib
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# ------------------------------------------------------------------ which kernels serve a solve
# The family table of test_oracle_matrix.py (written out by hand, not taken from the library's
# rule): tests assert the family each of their solves ran, so a change of plan fails them.
LINDX_COMPILED = {(2, 1), (2, 2), (3, 1), (4, 1), (4, 2), (4, 4), (5, 1), (6, 2), (8, 1), (8, 2),
                  (8, 4), (13, 3), (16, 1), (16, 2), (16, 4)}
NN_COMPILED = {(3, 1), (4, 2), (5, 1)}
# compiled LinDx shapes whose Riccati stage (C, c, F, f slabs of a warp, double-buffered) does
# not fit the 56 KB per-warp budget: every solve of these runs the group sweep
UNSTAGED = {torch.float64: {(6, 2), (8, 1), (8, 2), (8, 4), (13, 3), (16, 1), (16, 2), (16, 4)},
            torch.float32: {(8, 4), (13, 3), (16, 1), (16, 2), (16, 4)}}


def expected_family(ns, nc, dtype, box_global, nn=False):
    """The family of a LinDx (or, with ``nn``, NNDynamics) solve whose batch fits the group
    sweep's capacity."""
    if nn:
        return "nn" if (ns, nc) in NN_COMPILED else "nn_rt"
    if (ns, nc) not in LINDX_COMPILED:
        return "runtime"
    if (ns, nc) in UNSTAGED[dtype] or (nc > 1 and box_global):
        return "group"
    return "thread"


def family(info):
    """The family a solve ran, from its SolveInfo: runtime, nn, nn_rt, group or thread."""
    lib = importlib.import_module("differentiable-ilqr_b200._lib")
    p = info._problem[0]
    return {lib.DYN_LINDX_RT: "runtime", lib.DYN_NN: "nn", lib.DYN_NN_RT: "nn_rt"}.get(
        p.dynamics, "group" if p.group_sweep else "thread")


def golden(name):
    z = np.load(os.path.join(GOLDEN, name))
    return {k: torch.from_numpy(np.asarray(z[k])) for k in z.files}


def rel(a, b):
    a = a.detach().cpu().double()
    b = b.detach().cpu().double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-300))


def lindx_problem(ns, nc, T, B, dtype, seed=0):
    """SURVEY 8d config 5 generator."""
    g = torch.Generator().manual_seed(seed)
    n = ns + nc
    f64 = torch.float64
    A = torch.randn(T, B, n, n, generator=g, dtype=f64)
    C = A.transpose(2, 3) @ A + torch.eye(n, dtype=f64)
    c = torch.randn(T, B, n, generator=g, dtype=f64)
    F = torch.cat((torch.eye(ns, dtype=f64).expand(T - 1, B, ns, ns)
                   + 0.2 * torch.randn(T - 1, B, ns, ns, generator=g, dtype=f64) / ns ** 0.5,
                   torch.randn(T - 1, B, ns, nc, generator=g, dtype=f64) / ns ** 0.5), 3)
    f = 0.1 * torch.randn(T - 1, B, ns, generator=g, dtype=f64)
    x0 = torch.randn(B, ns, generator=g, dtype=f64)
    return [t.to(dtype).contiguous() for t in (C, c, F, f, x0)]


def env_problem(port, name, T, B, dtype, sigma=0.5, seed=0):
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    if name == "cartpole":
        pdx = port.CartpoleDx(dtype=dtype)
        r = (torch.rand(B, 4, generator=g, dtype=f64) * 2 - 1) * sigma
        x0 = torch.stack((r[:, 0], r[:, 1], torch.cos(r[:, 2]), torch.sin(r[:, 2]), r[:, 3]), 1)
    elif name == "rocket":
        pdx = port.RocketDx(dtype=dtype)
        qv = torch.cat((torch.ones(B, 1, dtype=f64), 0.1 * torch.randn(B, 3, generator=g, dtype=f64)), 1)
        x0 = torch.cat(((torch.rand(B, 3, generator=g, dtype=f64) * 2 - 1) * 15,
                        torch.rand(B, 3, generator=g, dtype=f64) * 2 - 1,
                        qv / qv.norm(dim=1, keepdim=True),
                        (torch.rand(B, 3, generator=g, dtype=f64) * 2 - 1) * 0.1), 1)
    else:
        pdx = port.PendulumDx(dtype=dtype)
        th = (torch.rand(B, generator=g, dtype=f64) - 0.5) * 3.14159
        w = torch.rand(B, generator=g, dtype=f64) * 2 - 1
        x0 = torch.stack((torch.cos(th), torch.sin(th), w), 1)
    q, p = pdx.get_true_obj()
    C = torch.diag(q)[None, None].repeat(T, B, 1, 1)
    c = p[None, None].repeat(T, B, 1)
    kw = dict(u_lower=pdx.lower, u_upper=pdx.upper, eps=pdx.mpc_eps,
              linesearch_decay=pdx.linesearch_decay,
              max_linesearch_iter=pdx.max_linesearch_iter)
    return pdx, x0.to(dtype), C, c, kw


class SoftCost(torch.nn.Module):
    """A convex, non-quadratic cost Module: 1/2 tau' (A'A + I) tau + p' tau + w sum log cosh(tau)."""

    def __init__(self, n, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.A = torch.nn.Parameter(0.3 * torch.randn(n, n, generator=g, dtype=torch.float64))
        self.p = torch.nn.Parameter(0.5 * torch.randn(n, generator=g, dtype=torch.float64))
        self.w = torch.nn.Parameter(torch.tensor(0.7, dtype=torch.float64))

    def forward(self, tau):
        Q = self.A.t() @ self.A + torch.eye(self.A.shape[0], dtype=tau.dtype, device=tau.device)
        return 0.5 * ((tau @ Q) * tau).sum(1) + (tau * self.p).sum(1) \
            + self.w * torch.log(torch.cosh(tau)).sum(1)


class SoftDyn(torch.nn.Module):
    """A smooth dynamics Module without grad_input: x' = x + dt (A x + B u + 0.3 tanh(W x))."""

    def __init__(self, ns, nc, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.A = torch.nn.Parameter(0.4 * torch.randn(ns, ns, generator=g, dtype=torch.float64))
        self.B = torch.nn.Parameter(torch.randn(ns, nc, generator=g, dtype=torch.float64))
        self.W = torch.nn.Parameter(0.5 * torch.randn(ns, ns, generator=g, dtype=torch.float64))

    def forward(self, x, u):
        return x + 0.1 * (x @ self.A.t() + u @ self.B.t() + 0.3 * torch.tanh(x @ self.W.t()))
