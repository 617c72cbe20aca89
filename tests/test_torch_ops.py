"""The drop-in boundary as north_star words it: torch custom ops (TORCH_LIBRARY(dilqr, ...),
csrc/torch_ops.cpp) over the C ABI, and the reference's UNMODIFIED caller running against
this package (dropin.install())."""
import importlib
import os
import sys

import pytest
import torch

from common import env_problem, lindx_problem, rel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"


@pytest.fixture(scope="module")
def ops():
    m = importlib.import_module("differentiable-ilqr_b200.torch_ops")
    m.load()
    return m


def test_ops_are_registered_with_the_dispatcher(ops):
    for name in ("mpc_solve", "dilqr_backward", "lqr_kkt_backward"):
        op = getattr(torch.ops.dilqr, name)
        assert "dilqr::" + name in str(op.default._schema)
    s = str(torch.ops.dilqr.mpc_solve.default._schema)
    assert "Tensor x_init, Tensor C, Tensor c, Tensor? F" in s and "int lqr_iter" in s


def test_ops_have_no_cpu_kernel(ops):
    """CPU tensors are refused by the dispatcher: there is no CPU implementation to fall to."""
    x0 = torch.zeros(2, 5, dtype=torch.float64)
    C, c = torch.eye(6, dtype=torch.float64), torch.zeros(6, dtype=torch.float64)
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.dilqr.mpc_solve(x0, C, c, None, None, None, torch.ones(4, dtype=torch.float64), 2,
                                  10, -1.0, 1.0, 3, 1e-4, 0.5, 2, 5, 1e-4, 0)


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "il_env.py")),
                    reason="the reference tree only exists in the build container")
def test_unmodified_reference_il_env_runs_against_the_package(monkeypatch):
    """/root/reference/il_env.py, byte for byte, with its imports (`from mpc_explicit import
    MPC`, `from env_dx import pendulum, cartpole`, il_env.py:5-9) resolved to this package:
    IL_Env.mpc (il_env.py:153-188) reaches our solver with the reference's own arguments.
    (Build container: no GPU, so the solve itself is intercepted; the arguments are not.)"""
    from unittest.mock import MagicMock
    dropin = importlib.import_module("differentiable-ilqr_b200.dropin")
    solver = importlib.import_module("differentiable-ilqr_b200._solver")
    lib = importlib.import_module("differentiable-ilqr_b200._lib")
    saved = {k: sys.modules.get(k) for k in list(dropin.ALIASES) + ["setproctitle", "ref_il_env"]}
    try:
        for k in dropin.ALIASES:
            sys.modules.pop(k, None)
        sys.modules.setdefault("setproctitle", MagicMock())
        dropin.install(force=True)
        spec = importlib.util.spec_from_file_location("ref_il_env", os.path.join(REF, "il_env.py"))
        ref = importlib.util.module_from_spec(spec)
        sys.dont_write_bytecode = True
        spec.loader.exec_module(ref)
        assert ref.MPC is importlib.import_module("differentiable-ilqr_b200.mpc_explicit").MPC
        e = ref.IL_Env("cartpole", lqr_iter=7, mpc_T=12)
        assert type(e.true_dx).__module__.startswith("differentiable-ilqr_b200")
        torch.manual_seed(0)
        x0 = e.sample_xinit(n_batch=3)
        q, p = e.true_dx.get_true_obj()
        # without a GPU the call must stop at the "no CPU path" guard of the solver ...
        with pytest.raises(lib.DilqrLibraryError):
            e.mpc(e.true_dx, x0, q, p)
        # ... and with the solve intercepted we see exactly what the reference handed over
        seen = {}

        def fake(x_init, C_, c_, dyn, n_state, n_ctrl, T, **kw):
            seen.update(kw, x_init=x_init, C=C_, c=c_, dyn=dyn, dims=(n_state, n_ctrl, T))
            raise KeyboardInterrupt

        monkeypatch.setattr(solver, "solve_mpc", fake)
        with pytest.raises(KeyboardInterrupt):
            e.mpc(e.true_dx, x0, q, p)
        assert seen["dims"] == (5, 1, 12) and seen["lqr_iter"] == 7
        assert tuple(seen["C"].shape) == (12, 3, 6, 6) and tuple(seen["c"].shape) == (12, 3, 6)
        assert torch.equal(seen["C"][4, 1], torch.diag(q))            # il_env.py:159-162
        assert seen["u_lower"] == -100.0 and seen["u_upper"] == 100.0
        assert seen["eps"] == e.true_dx.mpc_eps and seen["max_linesearch_iter"] == 2
        assert seen["dyn"].kind == lib.DYN_CARTPOLE
        assert seen["dyn"].params[:4] == [pytest.approx(v) for v in (9.8, 1.0, 0.1, 0.5)]
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.mark.gpu
def test_op_equals_module_env(ops, dilqr, port, dev):
    """torch.ops.dilqr.mpc_solve == mpc_explicit.MPC (same kernels, same order): outputs
    bitwise, registered autograd == the module's backward."""
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    lib = importlib.import_module("differentiable-ilqr_b200._lib")
    T, B = 25, 48
    pdx, x0, C, c, kw = env_problem(port, "cartpole", T, B, torch.float64, sigma=0.05)
    g = torch.Generator().manual_seed(3)
    gx = torch.randn(T, B, 5, generator=g, dtype=torch.float64).to(dev)
    gu = torch.randn(T, B, 1, generator=g, dtype=torch.float64).to(dev)
    th1 = pdx.params.to(dev).requires_grad_()
    C1, c1 = C.to(dev).requires_grad_(), c.to(dev).requires_grad_()
    x, u, costs, du, qp = torch.ops.dilqr.mpc_solve(
        x0.to(dev), C1, c1, None, None, None, th1, lib.DYN_CARTPOLE, T, pdx.lower, pdx.upper, 60, 1e-9,
        pdx.linesearch_decay, pdx.max_linesearch_iter, 5, 1e-4, 0)
    ((x * gx).sum() + (u * gu).sum()).backward()
    th2 = pdx.params.to(dev).requires_grad_()
    C2, c2 = C.to(dev).requires_grad_(), c.to(dev).requires_grad_()
    m = dilqr.mpc_explicit.MPC(5, 1, T, u_lower=pdx.lower, u_upper=pdx.upper, lqr_iter=60, eps=1e-9,
                               linesearch_decay=pdx.linesearch_decay,
                               max_linesearch_iter=pdx.max_linesearch_iter, verbose=-1,
                               exit_unconverged=False, detach_unconverged=False,
                               richardson_passes=ops.RICHARDSON_PASSES, richardson_tol=None)
    x2, u2, costs2 = m(x0.to(dev), dilqr.QuadCost(C2, c2), env.CartpoleDx(th2))
    ((x2 * gx).sum() + (u2 * gu).sum()).backward()
    assert torch.equal(x, x2) and torch.equal(u, u2) and torch.equal(costs, costs2)
    assert [v for v in qp.tolist() if v >= 0] == m.last_info.qp_iters
    assert rel(th1.grad, th2.grad) < 1e-12
    assert rel(C1.grad, C2.grad) < 1e-12 and rel(c1.grad, c2.grad) < 1e-12


@pytest.mark.gpu
def test_op_equals_module_rocket(ops, dilqr, port, dev):
    """The op plans its solve in the library like the Python binding, so a rocket batch (too
    large for one thread per problem) takes the group sweep -- two kernels per iteration -- in
    both, and the forward outputs agree bitwise.  Forward only: the op's registered backward has
    no rocket kernels."""
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    lib = importlib.import_module("differentiable-ilqr_b200._lib")
    T, B = 20, 64
    pdx, x0, C, c, kw = env_problem(port, "rocket", T, B, torch.float64)
    theta = pdx.params.to(dev)
    with torch.no_grad():
        x, u, costs, du, qp = torch.ops.dilqr.mpc_solve(
            x0.to(dev), C.to(dev), c.to(dev), None, None, None, theta, lib.DYN_ROCKET, T,
            pdx.lower, pdx.upper, 4, pdx.mpc_eps, pdx.linesearch_decay, pdx.max_linesearch_iter,
            5, 1e-4, 0)
        assert lib.lib().dilqr_last_iterate_launches() == 2
        m = dilqr.mpc_explicit.MPC(13, 3, T, u_lower=pdx.lower, u_upper=pdx.upper, lqr_iter=4,
                                   eps=pdx.mpc_eps, linesearch_decay=pdx.linesearch_decay,
                                   max_linesearch_iter=pdx.max_linesearch_iter, verbose=-1,
                                   exit_unconverged=False, detach_unconverged=False)
        x2, u2, costs2 = m(x0.to(dev), dilqr.QuadCost(C.to(dev), c.to(dev)), env.RocketDx(theta))
    assert torch.equal(x, x2) and torch.equal(u, u2) and torch.equal(costs, costs2)
    assert [v for v in qp.tolist() if v >= 0] == m.last_info.qp_iters


@pytest.mark.gpu
@pytest.mark.parametrize("boxed", [False, True])
def test_op_equals_module_lindx(ops, dilqr, dev, boxed):
    lib = importlib.import_module("differentiable-ilqr_b200._lib")
    ns, nc, T, B = 4, 2, 12, 40
    C, c, F, f, x0 = [t.to(dev) for t in lindx_problem(ns, nc, T, B, torch.float64, seed=2)]
    lo, hi = (-1.0, 1.0) if boxed else (None, None)
    outs = []
    for use_op in (True, False):
        leaves = [t.clone().requires_grad_() for t in (x0, C, c, F, f)]
        if use_op:
            x, u, costs, _, _ = torch.ops.dilqr.mpc_solve(
                leaves[0], leaves[1], leaves[2], leaves[3], leaves[4], None,
                torch.zeros(1, dtype=torch.float64), lib.DYN_LINDX, T, lo, hi, 10, 1e-7, 0.2, 10, 5,
                1e-4, 0)
        else:
            m = dilqr.MPC(ns, nc, T, u_lower=lo, u_upper=hi, lqr_iter=10, verbose=-1,
                          exit_unconverged=False, detach_unconverged=False)
            x, u, costs = m(leaves[0], dilqr.QuadCost(leaves[1], leaves[2]),
                            dilqr.LinDx(leaves[3], leaves[4]))
        (x.pow(2).sum() + u.sum()).backward()
        outs.append([x.detach(), u.detach()] + [t.grad for t in leaves])
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    for a, b in zip(outs[0][2:], outs[1][2:]):
        assert rel(a, b) < 1e-12


@pytest.mark.gpu
def test_opcheck(ops, port, dev):
    lib = importlib.import_module("differentiable-ilqr_b200._lib")
    pdx, x0, C, c, kw = env_problem(port, "pendulum", 10, 8, torch.float64, sigma=0.3)
    args = (x0.to(dev), C.to(dev), c.to(dev), None, None, None, pdx.params.to(dev),
            lib.DYN_PENDULUM, 10, pdx.lower, pdx.upper, 5, 1e-3, pdx.linesearch_decay,
            pdx.max_linesearch_iter, 5, 1e-4, 0)
    torch.library.opcheck(torch.ops.dilqr.mpc_solve.default, args,
                          test_utils=("test_schema", "test_faketensor"))
