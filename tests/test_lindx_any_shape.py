"""LinDx problems of any shape up to 32 variables: the runtime-dimension kernels
(DILQR_DYN_LINDX_RT, csrc/rt_kernels.cuh).

CPU tests check the ABI: which kernels the library picks for a shape, the range of the new
dynamics id and its argument checks.  GPU tests check that the runtime path computes what the
compiled kernels compute on the shapes both serve, that shapes without compiled kernels agree
with the CPU oracle, that their KKT gradients do, and that the user-level paths that used to
stop at "no kernel compiled" now run."""
import ctypes as C
import importlib

import pytest
import torch

from common import lindx_problem, rel


def _lib():
    return importlib.import_module("differentiable-ilqr_b200._lib")


# ------------------------------------------------------------------ CPU: the C ABI
def test_lindx_kernels_choice():
    lib = _lib()
    L = lib.lib()
    for dt in (lib.F32, lib.F64):
        for ns, nc in ((4, 2), (16, 4)):
            assert L.dilqr_lindx_kernels(dt, ns, nc) == lib.DYN_LINDX
        for ns, nc in ((7, 7), (7, 3), (6, 1), (24, 8)):
            assert L.dilqr_lindx_kernels(dt, ns, nc) == lib.DYN_LINDX_RT
        assert L.dilqr_lindx_kernels(dt, 24, 9) == -2
        assert L.dilqr_lindx_kernels(dt, 0, 2) == -1
        assert L.dilqr_lindx_kernels(dt, 3, 0) == -1
    assert L.dilqr_lindx_kernels(7, 4, 2) == -1


def test_supported_runtime_range():
    lib = _lib()
    L = lib.lib()
    for dt in (lib.F32, lib.F64):
        for ns, nc in ((4, 2), (7, 3), (31, 1)):
            assert L.dilqr_supported(dt, ns, nc, lib.DYN_LINDX_RT) == 1
        assert L.dilqr_supported(dt, 30, 3, lib.DYN_LINDX_RT) == 0
        assert L.dilqr_supported(dt, 0, 3, lib.DYN_LINDX_RT) == 0


def _aligned_buffer(n_doubles=4096):
    buf = (C.c_double * n_doubles)()
    base = C.addressof(buf)
    return buf, base + (-base) % 16


def test_plan_runtime_replays_trace():
    lib = _lib()
    L = lib.lib()
    s = lib.DilqrSolve()
    s.n_state, s.n_ctrl, s.T, s.n_batch, s.dtype = 8, 4, 10, 64, lib.F64
    s.dynamics, s.bounds_kind, s.solo = lib.DYN_LINDX_RT, lib.BOUNDS_SCALAR, 0
    s.group_sweep = 1
    assert L.dilqr_mpc_plan(C.byref(s)) == 0
    assert s.group_sweep == 0
    s.n_state = 29
    assert L.dilqr_mpc_plan(C.byref(s)) == -2


def test_runtime_argument_checks():
    lib = _lib()
    L = lib.lib()
    buf, base = _aligned_buffer()
    s = lib.DilqrSolve()
    s.n_state, s.n_ctrl, s.T, s.n_batch, s.dtype = 7, 3, 10, 4, lib.F64
    s.dynamics = lib.DYN_LINDX_RT
    s.x_init = s.C = s.c = base
    s.status = s.workspace = base
    s.workspace_bytes = 1 << 40
    assert L.dilqr_mpc_begin(C.byref(s), None) == -1          # LinDx without F
    s.F = base + 8
    assert L.dilqr_mpc_begin(C.byref(s), None) == -3          # misaligned F
    s.F = base
    s.workspace_bytes = 16
    assert L.dilqr_mpc_iterate(C.byref(s), None) == -4        # workspace too small
    s.n_state, s.n_ctrl = 30, 3                                # 33 variables
    s.workspace_bytes = 1 << 40
    assert L.dilqr_mpc_begin(C.byref(s), None) == -2
    assert L.dilqr_workspace_bytes(C.byref(s)) > 0
    s.n_state, s.n_ctrl = 7, 3
    assert L.dilqr_mpc_gains(C.byref(s), None, None) == -2    # as for LinDx
    k = lib.DilqrKkt()
    k.n_state, k.n_ctrl, k.T, k.n_batch, k.dtype = 30, 3, 10, 4, lib.F64
    k.C = k.c = k.F = k.x = k.u = k.dx = k.du = k.r = base
    k.dynamics = lib.DYN_LINDX_RT
    assert L.dilqr_kkt_grads(C.byref(k), None) == -2
    k.dynamics = 9
    assert L.dilqr_kkt_grads(C.byref(k), None) == -1


def test_out_of_range_message():
    """A shape beyond 32 variables still raises DilqrLibraryError, naming the limit."""
    lib = _lib()
    sol = importlib.import_module("differentiable-ilqr_b200._solver")
    with pytest.raises(lib.DilqrLibraryError, match="32 variables"):
        sol.lindx_kernels(torch.float64, 30, 3)
    assert sol.lindx_kernels(torch.float64, 7, 3) == lib.DYN_LINDX_RT
    assert sol.lindx_kernels(torch.float32, 4, 2) == lib.DYN_LINDX


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def sol():
    return importlib.import_module("differentiable-ilqr_b200._solver")


# The cases of the cross-check: DilqrSolve options the LinDx path honours.  Each is
# (name, B, options); `bounds` "scalar" / "tensor" / None.
CASES = [
    ("free", 33, dict()),
    ("scalar_box", 1, dict(bounds="scalar")),
    ("tensor_box", 33, dict(bounds="tensor")),
    ("u_zero_I", 33, dict(zero_I=True)),
    ("delta_u", 33, dict(bounds="scalar", delta_u=0.3)),
    ("solo1", 33, dict(bounds="scalar", solo=1)),
    ("solo2", 33, dict(bounds="scalar", solo=2)),
    ("C_bcast1", 33, dict(bounds="scalar", bcast=1)),
    ("C_bcast2", 1, dict(bcast=2)),
    ("no_f", 33, dict(bounds="scalar", no_f=True)),
    ("chol_reg", 33, dict(gain_solve=1)),
]


def _case_inputs(ns, nc, T, B, dtype, opt, seed):
    C_, c_, F, f, x0 = lindx_problem(ns, nc, T, B, dtype, seed=seed)
    kw = {}
    if opt.get("bounds") == "scalar":
        kw.update(u_lower=-1.0, u_upper=1.0)
    elif opt.get("bounds") == "tensor":
        g = torch.Generator().manual_seed(seed + 1)
        lo = -0.5 - torch.rand(T, B, nc, generator=g, dtype=torch.float64)
        kw.update(u_lower=lo.to(dtype), u_upper=(-lo).to(dtype))
    if opt.get("zero_I"):
        g = torch.Generator().manual_seed(seed + 2)
        kw["u_zero_I"] = torch.rand(T, B, nc, generator=g) < 0.3
    if "delta_u" in opt:
        kw["delta_u"] = opt["delta_u"]
    if opt.get("bcast") == 1:
        C_, c_ = C_[:, 0].contiguous(), c_[:, 0].contiguous()
    elif opt.get("bcast") == 2:
        C_, c_ = C_[0, 0].contiguous(), c_[0, 0].contiguous()
    if opt.get("no_f"):
        f = None
    return C_, c_, F, f, x0, kw


def _solve(sol, kind, ns, nc, T, inputs, opt, dev, step):
    C_, c_, F, f, x0, kw = inputs
    lib = _lib()
    kw = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in kw.items()}
    dyn = sol.DynSpec(kind, F=F.to(dev), f=None if f is None else f.to(dev))
    Cd, cd = C_.to(dev), c_.to(dev)   # [n,n] / [T,n,n] select the broadcast cost layouts
    extra = dict(solo=opt.get("solo", 0), gain_solve=opt.get("gain_solve", lib.GAIN_PLAIN))
    if step:
        g = torch.Generator().manual_seed(7)
        u0 = (0.3 * torch.randn(T, x0.shape[0], nc, generator=g, dtype=torch.float64)).to(x0.dtype)
        port = importlib.import_module("port")
        xc = port.get_traj(T, u0, x0, port.LinDx(F, f))
        return sol.solve_mpc(x0.to(dev), Cd, cd, dyn, ns, nc, T, u_init=u0.to(dev), x_cur=xc.to(dev),
                             want_gains=True, verbose=-1, **extra, **kw)
    return sol.solve_mpc(x0.to(dev), Cd, cd, dyn, ns, nc, T, lqr_iter=10, verbose=-1, **extra, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("step", [True, False], ids=["lqr_step", "mpc10"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("ns,nc", [(2, 1), (3, 1), (4, 2), (4, 4), (5, 1), (8, 4), (13, 3), (16, 4)])
def test_runtime_equals_compiled(sol, dev, ns, nc, dtype, step):
    """DYN_LINDX_RT against DYN_LINDX on compiled shapes.  Every entry is formed by the same
    operations in the same order, so the two agree to round-off; where the compiled path runs
    the group sweep (its own association), to 1e-9 with identical pnqp counts."""
    lib = _lib()
    T = 7
    for i, (name, B, opt) in enumerate(CASES):
        if name == "chol_reg" and nc == 1:
            continue
        inputs = _case_inputs(ns, nc, T, B, dtype, opt, seed=100 + i)
        xa, ua, ca, ia = _solve(sol, lib.DYN_LINDX, ns, nc, T, inputs, opt, dev, step)
        xb, ub, cb, ib = _solve(sol, lib.DYN_LINDX_RT, ns, nc, T, inputs, opt, dev, step)
        assert ia._problem[0].dynamics == lib.DYN_LINDX and ib._problem[0].dynamics == lib.DYN_LINDX_RT
        group = bool(ia._problem[0].group_sweep)
        tol = (1e-9 if group else 1e-12) if dtype == torch.float64 else 1e-5
        what = "%s B=%d group_sweep=%d" % (name, B, group)
        assert rel(xb, xa) <= tol and rel(ub, ua) <= tol and rel(cb, ca) <= tol, what
        assert ib.qp_iters == ia.qp_iters and ib.n_iters == ia.n_iters, what
        if step:
            assert rel(ib.K, ia.K) <= tol and rel(ib.k, ia.k) <= tol, what
            if not group:
                assert torch.equal(ib.alphas, ia.alphas), what


def _oracle_cases():
    out = []
    for ns, nc in ((1, 1), (6, 1), (7, 3), (3, 5), (10, 6), (24, 8), (31, 1)):
        for T, B in ((2, 1), (12, 33), (30, 100)):
            for boxed in (False, True):
                out.append((ns, nc, T, B, boxed))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("ns,nc,T,B,boxed", _oracle_cases())
def test_uncompiled_shape_vs_oracle(sol, dev, ns, nc, T, B, boxed, dtype):
    """One LQRStep of a shape with no compiled kernels against the CPU oracle (the
    tolerances of test_gpu_parity.test_lindx_single_step)."""
    port = importlib.import_module("port")
    lib = _lib()
    assert lib.lib().dilqr_lindx_kernels(sol._DT[dtype], ns, nc) == lib.DYN_LINDX_RT
    C_, c_, F, f, x0 = lindx_problem(ns, nc, T, B, dtype)
    kw = dict(u_lower=-1.0, u_upper=1.0) if boxed else {}
    u0 = torch.zeros(T, B, nc, dtype=dtype)
    xc = port.get_traj(T, u0, x0, port.LinDx(F, f))
    o = port.lqr_step(x0, C_, c_, F, xc, u0, port.QuadCost(C_, c_), port.LinDx(F, f), ns, nc, **kw)
    dyn = sol.DynSpec(lib.DYN_LINDX, F=F.to(dev), f=f.to(dev))
    x, u, costs, info = sol.solve_mpc(x0.to(dev), C_.to(dev), c_.to(dev), dyn, ns, nc, T,
                                      u_init=u0.to(dev), x_cur=xc.to(dev), want_gains=True,
                                      verbose=-1, **kw)
    assert info._problem[0].dynamics == lib.DYN_LINDX_RT
    tol = 3e-9 if dtype == torch.float64 else 3e-4
    assert rel(x, o.x) < tol and rel(u, o.u) < tol and rel(costs, o.costs) < tol
    assert rel(info.K, torch.stack(o.Ks[::-1])) < tol and rel(info.k, torch.stack(o.ks[::-1])) < tol
    assert rel(info.alphas, o.alphas) == 0.0
    if dtype == torch.float64:
        assert info.qp_iters[0] == o.n_total_qp_iter


@pytest.mark.gpu
@pytest.mark.parametrize("boxed", [False, True])
@pytest.mark.parametrize("ns,nc", [(7, 3), (24, 8)])
def test_kkt_gradients_vs_oracle(ns, nc, boxed, dev):
    """mpc.MPC + .backward() on runtime shapes: dx0, dC, dc, dF, df against port.kkt_backward
    at the same solution."""
    dilqr = importlib.import_module("differentiable-ilqr_b200")
    port = importlib.import_module("port")
    T, B = 10, 9
    C_, c_, F, f, x0 = lindx_problem(ns, nc, T, B, torch.float64, seed=4)
    kw = dict(u_lower=-1.0, u_upper=1.0) if boxed else {}
    m = dilqr.MPC(ns, nc, T, lqr_iter=20, verbose=-1, exit_unconverged=False,
                  detach_unconverged=False, **kw)
    leaves = [t.to(dev).requires_grad_() for t in (x0, C_, c_, F, f)]
    x, u, _ = m(leaves[0], dilqr.QuadCost(leaves[1], leaves[2]), dilqr.LinDx(leaves[3], leaves[4]))
    g = torch.Generator().manual_seed(12)
    gx = torch.randn(x.shape, generator=g, dtype=torch.float64)
    gu = torch.randn(u.shape, generator=g, dtype=torch.float64)
    ((x * gx.to(dev)).sum() + (u * gu.to(dev)).sum()).backward()
    k = port.kkt_backward(gx, gu, x0, C_, c_, F, f, x.detach().cpu(), u.detach().cpu(), ns, nc, **kw)
    for leaf, ref_, nm in zip(leaves, (k.dx_init, k.dC, k.dc, k.dF, k.df), ("dx0", "dC", "dc", "dF", "df")):
        assert rel(leaf.grad, ref_) < 1e-10, nm


@pytest.mark.gpu
def test_slew_rate_5p1(dev):
    """slew_rate_penalty on a 5+1 LinDx augments the state to 6+1, a shape with no compiled
    kernels; against the oracle on the same augmented problem."""
    dilqr = importlib.import_module("differentiable-ilqr_b200")
    port = importlib.import_module("port")
    ns, nc, T, B, gam = 5, 1, 12, 9, 0.5
    C_, c_, F, f, x0 = lindx_problem(ns, nc, T, B, torch.float64, seed=5)
    m = dilqr.MPC(ns, nc, T, u_lower=-1.0, u_upper=1.0, lqr_iter=20, verbose=-1,
                  exit_unconverged=False, slew_rate_penalty=gam)
    x, u, costs = m(x0.to(dev), dilqr.QuadCost(C_.to(dev), c_.to(dev)), dilqr.LinDx(F.to(dev), f.to(dev)))
    n, nt = ns + nc, ns + 2 * nc
    gI = gam * torch.eye(nc, dtype=torch.float64)
    Ca = torch.zeros(T, B, nt, nt, dtype=torch.float64)
    Ca[:, :, :nc, :nc] = gI
    Ca[:, :, -nc:, :nc] = -gI
    Ca[:, :, :nc, -nc:] = -gI
    Ca[:, :, -nc:, -nc:] = gI
    Ca = Ca + torch.nn.functional.pad(C_, (nc, 0, nc, 0))
    ca = torch.cat((torch.zeros(T, B, nc, dtype=torch.float64), c_), 2)
    F0 = torch.cat((torch.zeros(nc, n, dtype=torch.float64), torch.eye(nc, dtype=torch.float64)), 1)
    Fa = torch.cat((F0.expand(T - 1, B, nc, nt), torch.cat((torch.zeros(T - 1, B, ns, nc,
                                                                         dtype=torch.float64), F), 3)), 2)
    fa = torch.cat((torch.zeros(T - 1, B, nc, dtype=torch.float64), f), 2)
    xa0 = torch.cat((torch.zeros(B, nc, dtype=torch.float64), x0), 1)
    o = port.mpc_forward(xa0, port.QuadCost(Ca, ca), port.LinDx(Fa, fa), ns + nc, nc, T,
                         u_lower=-1.0, u_upper=1.0, lqr_iter=20, final_pass=False)
    # later iterations of a cold-start solve amplify last-bit differences of the sums into
    # different pnqp paths, so beyond the first step only the solution is compared (as in
    # test_gpu_parity.test_affine_dynamics_and_slew_rate_golden)
    assert m.last_info.qp_iters[0] == o.qp_iters[0]
    assert rel(x, o.x[:, :, nc:]) < 1e-8 and rel(u, o.u) < 1e-8 and rel(costs, o.costs) < 1e-9


@pytest.mark.gpu
def test_affine_dynamics_7p3(dev):
    dilqr = importlib.import_module("differentiable-ilqr_b200")
    port = importlib.import_module("port")
    ns, nc, T, B = 7, 3, 10, 9
    C_, c_, _, _, x0 = lindx_problem(ns, nc, T, B, torch.float64, seed=6)
    g = torch.Generator().manual_seed(6)
    A = torch.eye(ns, dtype=torch.float64) + 0.1 * torch.randn(ns, ns, generator=g, dtype=torch.float64)
    Bm = 0.3 * torch.randn(ns, nc, generator=g, dtype=torch.float64)
    cv = 0.1 * torch.randn(ns, generator=g, dtype=torch.float64)
    m = dilqr.MPC(ns, nc, T, u_lower=-1.0, u_upper=1.0, lqr_iter=20, verbose=-1, exit_unconverged=False)
    x, u, costs = m(x0.to(dev), dilqr.QuadCost(C_.to(dev), c_.to(dev)),
                    dilqr.AffineDynamics(A.to(dev), Bm.to(dev), cv.to(dev)))
    F = torch.cat((A, Bm), 1).expand(T - 1, B, ns, ns + nc)
    f = cv.expand(T - 1, B, ns)
    o = port.mpc_forward(x0, port.QuadCost(C_, c_), port.LinDx(F, f), ns, nc, T, u_lower=-1.0,
                         u_upper=1.0, lqr_iter=20, final_pass=False)
    assert m.last_info.qp_iters[0] == o.qp_iters[0]   # later iterations: see test_slew_rate_5p1
    assert rel(x, o.x) < 1e-8 and rel(u, o.u) < 1e-8 and rel(costs, o.costs) < 1e-9


@pytest.mark.gpu
def test_module_cost_7p3(dev):
    """A Module cost on a 7+3 LinDx runs every LQR step through the LinDx sweep of its shape
    (mpc.py _forward_generic); a quadratic Module equals the QuadCost solve."""
    dilqr = importlib.import_module("differentiable-ilqr_b200")
    port = importlib.import_module("port")
    ns, nc, T, B = 7, 3, 8, 5
    n = ns + nc
    C_, c_, F, f, x0 = lindx_problem(ns, nc, T, B, torch.float64, seed=7)
    Cs, cs = C_[0, 0], c_[0, 0]

    class Quad(torch.nn.Module):
        def forward(self, tau):
            return 0.5 * ((tau @ Cs.to(tau.device)) * tau).sum(-1) + tau @ cs.to(tau.device)

    m = dilqr.MPC(ns, nc, T, u_lower=-1.0, u_upper=1.0, lqr_iter=10, verbose=-1,
                  exit_unconverged=False, n_batch=B)
    x, u, costs = m(x0.to(dev), Quad(), dilqr.LinDx(F.to(dev), f.to(dev)))
    Cd = Cs.expand(T, B, n, n).contiguous()
    cd = cs.expand(T, B, n).contiguous()
    o = port.mpc_forward(x0, port.QuadCost(Cd, cd), port.LinDx(F, f), ns, nc, T, u_lower=-1.0,
                         u_upper=1.0, lqr_iter=10, final_pass=False)
    assert rel(x, o.x) < 1e-8 and rel(u, o.u) < 1e-8


@pytest.mark.gpu
def test_lqr_step_7p3(dev):
    dilqr = importlib.import_module("differentiable-ilqr_b200")
    port = importlib.import_module("port")
    ns, nc, T, B = 7, 3, 12, 16
    C_, c_, F, f, x0 = lindx_problem(ns, nc, T, B, torch.float64, seed=3)
    u0 = 0.1 * torch.ones(T, B, nc, dtype=torch.float64)
    xc = port.get_traj(T, u0, x0, port.LinDx(F, f))
    kw = dict(u_lower=-1.0, u_upper=1.0)
    o = port.lqr_step(x0, C_, c_, F, xc, u0, port.QuadCost(C_, c_), port.LinDx(F, f), ns, nc, **kw)
    leaves = [t.to(dev).requires_grad_() for t in (x0, C_, c_, F, f)]
    step = dilqr.LQRStep(ns, nc, T, true_cost=dilqr.QuadCost(leaves[1], leaves[2]),
                         true_dynamics=dilqr.LinDx(leaves[3], leaves[4]), current_x=xc.to(dev),
                         current_u=u0.to(dev), **kw)
    x, u, n_qp, costs, du, mean_alpha = step(*leaves)
    assert rel(x, o.x) < 3e-9 and rel(u, o.u) < 3e-9 and rel(costs, o.costs) < 3e-9
    assert float(n_qp) == o.n_total_qp_iter
    g = torch.Generator().manual_seed(11)
    gx = torch.randn(x.shape, generator=g, dtype=torch.float64)
    gu = torch.randn(u.shape, generator=g, dtype=torch.float64)
    ((x * gx.to(dev)).sum() + (u * gu.to(dev)).sum()).backward()
    k = port.kkt_backward(gx, gu, x0, C_, c_, F, f, o.x, o.u, ns, nc, **kw)
    for leaf, ref_ in zip(leaves, (k.dx_init, k.dC, k.dc, k.dF, k.df)):
        assert rel(leaf.grad, ref_) < 1e-9


@pytest.mark.gpu
def test_torch_ops_7p3(sol, dev):
    """torch.ops.dilqr.mpc_solve + lqr_kkt_backward on 7+3, bitwise equal to the Python path."""
    ops = importlib.import_module("differentiable-ilqr_b200.torch_ops")
    ops.load()
    lib = _lib()
    ns, nc, T, B = 7, 3, 10, 9
    C_, c_, F, f, x0 = lindx_problem(ns, nc, T, B, torch.float64, seed=8)
    C_, c_, F, f, x0 = (t.to(dev) for t in (C_, c_, F, f, x0))
    x, u, costs, du, qp = torch.ops.dilqr.mpc_solve(
        x0, C_, c_, F, f, None, torch.zeros(1, dtype=torch.float64), lib.DYN_LINDX, T, -1.0, 1.0, 10,
        1e-7, 0.2, 10, 5, 1e-4, 0)
    x2, u2, c2, info = sol.solve_mpc(x0, C_, c_, sol.DynSpec(lib.DYN_LINDX, F=F, f=f), ns, nc, T,
                                     u_lower=-1.0, u_upper=1.0, lqr_iter=10, verbose=-1)
    assert torch.equal(x, x2) and torch.equal(u, u2) and torch.equal(costs, c2)
    assert [v for v in qp.tolist() if v >= 0] == info.qp_iters
    g = torch.Generator().manual_seed(9)
    gx = torch.randn(T, B, ns, generator=g, dtype=torch.float64).to(dev)
    gu = torch.randn(T, B, nc, generator=g, dtype=torch.float64).to(dev)
    a = torch.ops.dilqr.lqr_kkt_backward(gx, gu, x0, C_, c_, F, x, u, -1.0, 1.0)
    b = sol.kkt_backward(gx, gu, x0, C_, c_, F, f, x, u, ns, nc, u_lower=-1.0, u_upper=1.0)
    for ta, tb, nm in zip(a, b, ("dx0", "dC", "dc", "dF", "df")):
        assert torch.equal(ta, tb), nm


@pytest.mark.gpu
def test_scale_7p3_solo2(sol, dev):
    """7+3 boxed, T = 50, B = 65536 + 5, solo = 2: every problem is its own batch of one, so
    the first 64 problems of the full batch equal a B = 64 solve of those problems."""
    lib = _lib()
    ns, nc, T, B = 7, 3, 50, 65536 + 5
    C_, c_, F, f, x0 = lindx_problem(ns, nc, T, 64, torch.float64, seed=10)
    reps = (B + 63) // 64
    g = torch.Generator(device=dev).manual_seed(13)
    # the first 64 problems are the B = 64 batch; the others are perturbed copies of it
    Cb = C_.to(dev).repeat(1, reps, 1, 1)[:, :B].contiguous()
    Fb = F.to(dev).repeat(1, reps, 1, 1)[:, :B].contiguous()
    fb = f.to(dev).repeat(1, reps, 1)[:, :B].contiguous()
    cb = c_.to(dev).repeat(1, reps, 1)[:, :B].contiguous()
    cb[:, 64:] += torch.randn(cb[:, 64:].shape, generator=g, device=dev, dtype=cb.dtype)
    xb = x0.to(dev).repeat(reps, 1)[:B].contiguous()
    xb[64:] += torch.randn(xb[64:].shape, generator=g, device=dev, dtype=xb.dtype)
    kw = dict(u_lower=-1.0, u_upper=1.0, lqr_iter=10, verbose=-1, solo=2)
    X, U, Cst, _ = sol.solve_mpc(xb, Cb, cb, sol.DynSpec(lib.DYN_LINDX, F=Fb, f=fb), ns, nc, T, **kw)
    torch.cuda.synchronize()
    x, u, cst, _ = sol.solve_mpc(xb[:64], Cb[:, :64], cb[:, :64],
                                 sol.DynSpec(lib.DYN_LINDX, F=Fb[:, :64], f=fb[:, :64]), ns, nc, T, **kw)
    assert torch.isfinite(X).all() and torch.isfinite(U).all()
    assert rel(X[:, :64], x) <= 1e-12 and rel(U[:, :64], u) <= 1e-12 and rel(Cst[:64], cst) <= 1e-12
