"""NNDynamics problems of any shape up to 32 variables: the runtime-dimension network kernels
(DILQR_DYN_NN_RT, csrc/rt_kernels.cuh).

CPU tests check the ABI: which kernels the library picks for a network of a given shape, the
range of the new dynamics id and its argument checks.  GPU tests check that the runtime path
computes what the compiled network kernels compute on the shapes both serve, that shapes without
compiled kernels agree with the CPU oracle and with the torch path of mpc.MPC, that gradients
through mpc.MPC are right, and that a large solo = 2 batch equals a small one."""
import ctypes as C
import importlib

import pytest
import torch

from common import lindx_problem, rel


def _lib():
    return importlib.import_module("differentiable-ilqr_b200._lib")


# ------------------------------------------------------------------ CPU: the C ABI
def test_nn_kernels_choice():
    lib = _lib()
    L = lib.lib()
    for dt in (lib.F32, lib.F64):
        for ns, nc in ((3, 1), (4, 2), (5, 1)):
            assert L.dilqr_nn_kernels(dt, ns, nc) == lib.DYN_NN
        for ns, nc in ((1, 1), (6, 2), (7, 3), (31, 1)):
            assert L.dilqr_nn_kernels(dt, ns, nc) == lib.DYN_NN_RT
        assert L.dilqr_nn_kernels(dt, 24, 9) == -2
        assert L.dilqr_nn_kernels(dt, 0, 2) == -1
        assert L.dilqr_nn_kernels(dt, 3, 0) == -1
    assert L.dilqr_nn_kernels(7, 3, 1) == -1


def test_supported_and_plan_runtime_range():
    lib = _lib()
    L = lib.lib()
    for dt in (lib.F32, lib.F64):
        for ns, nc in ((3, 1), (1, 1), (7, 3), (31, 1)):
            assert L.dilqr_supported(dt, ns, nc, lib.DYN_NN_RT) == 1
        assert L.dilqr_supported(dt, 30, 3, lib.DYN_NN_RT) == 0
        assert L.dilqr_supported(dt, 0, 3, lib.DYN_NN_RT) == 0
        # the meaning of DYN_NN does not change: compiled shapes only
        assert L.dilqr_supported(dt, 7, 3, lib.DYN_NN) == 0
    s = lib.DilqrSolve()
    s.n_state, s.n_ctrl, s.T, s.n_batch, s.dtype = 6, 2, 10, 64, lib.F64
    s.dynamics, s.bounds_kind, s.solo = lib.DYN_NN_RT, lib.BOUNDS_SCALAR, 0
    s.group_sweep = 1
    assert L.dilqr_mpc_plan(C.byref(s)) == 0
    assert s.group_sweep == 0
    s.n_state = 31
    assert L.dilqr_mpc_plan(C.byref(s)) == -2


def _aligned_buffer(n_doubles=4096):
    buf = (C.c_double * n_doubles)()
    base = C.addressof(buf)
    return buf, base + (-base) % 16


def test_runtime_argument_checks():
    lib = _lib()
    L = lib.lib()
    buf, base = _aligned_buffer()
    s = lib.DilqrSolve()
    s.n_state, s.n_ctrl, s.T, s.n_batch, s.dtype = 7, 3, 10, 4, lib.F64
    s.dynamics = lib.DYN_NN_RT
    s.x_init = s.C = s.c = base
    s.status = s.workspace = base
    s.workspace_bytes = 1 << 40
    s.dyn_ai[0], s.dyn_ai[1], s.dyn_ai[2], s.dyn_ai[3] = 16, 0, 1, 0
    assert L.dilqr_mpc_begin(C.byref(s), None) == -1          # no weights
    s.dyn_aux = base
    s.dyn_ai[0] = 129 | (6 << 16)                             # two layers, H1 > 128
    assert L.dilqr_mpc_begin(C.byref(s), None) == -1
    s.dyn_ai[0] = 128 | (6 << 16)
    s.dyn_ai[1] = 2                                           # activation
    assert L.dilqr_mpc_begin(C.byref(s), None) == -1
    s.dyn_ai[1], s.dyn_ai[3] = 1, 2                           # linearisation
    assert L.dilqr_mpc_begin(C.byref(s), None) == -1
    s.dyn_ai[3] = 1
    s.workspace_bytes = 16
    assert L.dilqr_mpc_iterate(C.byref(s), None) == -4        # workspace too small
    s.workspace_bytes = 1 << 40
    assert L.dilqr_mpc_gains(C.byref(s), None, None) == -2    # as for DYN_NN
    k = lib.DilqrKkt()
    k.n_state, k.n_ctrl, k.T, k.n_batch, k.dtype = 7, 3, 10, 4, lib.F64
    k.C = k.c = k.F = k.x = k.u = k.dx = k.du = k.r = base
    k.dynamics = lib.DYN_NN_RT                                # the NN backward is a LinDx problem
    assert L.dilqr_kkt_grads(C.byref(k), None) == -1


def test_out_of_range_message():
    lib = _lib()
    sol = importlib.import_module("differentiable-ilqr_b200._solver")
    with pytest.raises(lib.DilqrLibraryError, match="32 variables"):
        sol.nn_kernels(torch.float64, 30, 3)
    assert sol.nn_kernels(torch.float64, 7, 3) == lib.DYN_NN_RT
    assert sol.nn_kernels(torch.float32, 4, 2) == lib.DYN_NN


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def sol():
    return importlib.import_module("differentiable-ilqr_b200._solver")


@pytest.fixture(scope="module")
def dilqr():
    return importlib.import_module("differentiable-ilqr_b200")


@pytest.fixture(scope="module")
def port():
    return importlib.import_module("port")


def _net(dilqr, ns, nc, hidden, act, seed):
    """A seeded NNDynamics (float64, CPU) whose rollouts stay bounded over the horizons used."""
    g = torch.Generator().manual_seed(seed)
    net = dilqr.NNDynamics(ns, nc, hidden_sizes=hidden, activation=act, passthrough=True).double()
    with torch.no_grad():
        for fc in net.fcs:
            fan_in = fc.weight.shape[1]
            fc.weight.copy_(torch.randn(fc.weight.shape, generator=g, dtype=torch.float64) / fan_in ** 0.5)
            fc.bias.copy_(0.1 * torch.randn(fc.bias.shape, generator=g, dtype=torch.float64))
        net.fcs[-1].weight.mul_(0.3)
    return net


def _rollout(net, x0, u):
    xs = [x0]
    with torch.no_grad():
        for t in range(u.shape[0] - 1):
            xs.append(net(xs[t], u[t]))
    return torch.stack(xs, 0)


# The options of the runtime-vs-compiled check: those of test_lindx_any_shape.CASES that apply
# to a network ("no_f" has no meaning without f).  (name, B, options)
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
    ("chol_reg", 33, dict(gain_solve=1)),
]

NETS = [(h, act, fd) for h in ([12], [40], [10, 6]) for act in ("sigmoid", "relu") for fd in (0, 1)]


def _case_inputs(ns, nc, T, B, dtype, opt, seed):
    C_, c_, _, _, x0 = lindx_problem(ns, nc, T, B, dtype, seed=seed)
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
    return C_, c_, x0, kw


def _solve(sol, kind, net, fd, ns, nc, T, inputs, opt, dev, step):
    C_, c_, x0, kw = inputs
    lib = _lib()
    dtype = x0.dtype
    kw = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in kw.items()}
    aux, ai = net._dilqr_pack(dtype, dev)
    ai[3] = fd
    dyn = sol.DynSpec(kind, aux=aux, ai=ai)
    extra = dict(solo=opt.get("solo", 0), gain_solve=opt.get("gain_solve", lib.GAIN_PLAIN))
    if step:
        g = torch.Generator().manual_seed(7)
        u0 = 0.3 * torch.randn(T, x0.shape[0], nc, generator=g, dtype=torch.float64)
        xc = _rollout(net, x0.double(), u0)
        return sol.solve_mpc(x0.to(dev), C_.to(dev), c_.to(dev), dyn, ns, nc, T,
                             u_init=u0.to(dtype).to(dev), x_cur=xc.to(dtype).to(dev),
                             want_gains=True, verbose=-1, **extra, **kw)
    return sol.solve_mpc(x0.to(dev), C_.to(dev), c_.to(dev), dyn, ns, nc, T, lqr_iter=10,
                         verbose=-1, **extra, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("step", [True, False], ids=["lqr_step", "mpc10"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("hidden,act,fd", NETS)
@pytest.mark.parametrize("ns,nc", [(3, 1), (4, 2), (5, 1)])
def test_runtime_equals_compiled(sol, dilqr, dev, ns, nc, hidden, act, fd, dtype, step):
    """DYN_NN_RT against DYN_NN on the compiled shapes: the network values and the Riccati
    update are formed by the same operations in the same order, so the two agree to round-off
    with identical pnqp counts, iteration counts and line-search steps."""
    lib = _lib()
    T = 7
    net = _net(dilqr, ns, nc, hidden, act, seed=20 + len(hidden))
    for i, (name, B, opt) in enumerate(CASES):
        if name == "chol_reg" and nc == 1:
            continue
        inputs = _case_inputs(ns, nc, T, B, dtype, opt, seed=100 + i)
        xa, ua, ca, ia = _solve(sol, lib.DYN_NN, net, fd, ns, nc, T, inputs, opt, dev, step)
        xb, ub, cb, ib = _solve(sol, lib.DYN_NN_RT, net, fd, ns, nc, T, inputs, opt, dev, step)
        assert ia._problem[0].dynamics == lib.DYN_NN and ib._problem[0].dynamics == lib.DYN_NN_RT
        tol = 1e-12 if dtype == torch.float64 else 1e-5
        what = "%s B=%d" % (name, B)
        assert rel(xb, xa) <= tol and rel(ub, ua) <= tol and rel(cb, ca) <= tol, what
        assert ib.qp_iters == ia.qp_iters and ib.n_iters == ia.n_iters, what
        if step:
            assert rel(ib.K, ia.K) <= tol and rel(ib.k, ia.k) <= tol, what
            assert torch.equal(ib.alphas, ia.alphas), what


def _oracle_cases():
    out = []
    for ns, nc in ((1, 1), (2, 1), (6, 2), (7, 3), (12, 4), (24, 8), (31, 1)):
        for H in (7, 40):
            for act in ("sigmoid", "relu"):
                for boxed in (False, True):
                    out.append((ns, nc, H, act, boxed))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("ns,nc,H,act,boxed", _oracle_cases())
def test_uncompiled_shape_vs_oracle(sol, dilqr, port, dev, ns, nc, H, act, boxed, dtype):
    """One LQR step (the begin rollout, the Riccati sweep with the network's Jacobians, the
    line search through the network) of a shape with no compiled kernels against the CPU
    oracle (the tolerances of test_lindx_any_shape.test_uncompiled_shape_vs_oracle)."""
    lib = _lib()
    T, B = 10, 17
    assert lib.lib().dilqr_nn_kernels(sol._DT[dtype], ns, nc) == lib.DYN_NN_RT
    net = _net(dilqr, ns, nc, [H], act, seed=ns * 100 + nc + H)
    C_, c_, _, _, x0 = lindx_problem(ns, nc, T, B, dtype, seed=ns + nc)
    kw = dict(u_lower=-1.0, u_upper=1.0) if boxed else {}
    W1, b1, W2, b2 = (p.detach().to(dtype) for fc in net.fcs for p in (fc.weight, fc.bias))
    o = port.mpc_forward(x0, port.QuadCost(C_, c_), port.NNDynamics(W1, b1, W2, b2, act), ns, nc,
                         T, lqr_iter=1, final_pass=False, **kw)
    aux, ai = net._dilqr_pack(dtype, dev)
    x, u, costs, info = sol.solve_mpc(x0.to(dev), C_.to(dev), c_.to(dev),
                                      sol.DynSpec(lib.DYN_NN, aux=aux, ai=ai), ns, nc, T,
                                      lqr_iter=1, verbose=-1, **kw)
    assert info._problem[0].dynamics == lib.DYN_NN_RT
    tol = 3e-9 if dtype == torch.float64 else 3e-4
    assert rel(x, o.x) < tol and rel(u, o.u) < tol and rel(costs, o.costs) < tol
    if dtype == torch.float64:
        assert info.qp_iters == o.qp_iters


def _torch_path(monkeypatch, dilqr):
    def refuse(self, dtype, device):
        raise NotImplementedError("forced torch path")
    monkeypatch.setattr(dilqr.NNDynamics, "_dilqr_pack", refuse)


@pytest.mark.gpu
@pytest.mark.parametrize("fd", [False, True], ids=["analytic", "finite_diff"])
@pytest.mark.parametrize("hidden", [[10, 6], [128, 16]])
@pytest.mark.parametrize("ns,nc", [(6, 2), (12, 4)])
def test_two_layers_and_fd_vs_torch_path(dilqr, dev, monkeypatch, ns, nc, hidden, fd):
    """Two hidden layers and the central-difference linearisation on uncompiled shapes: one LQR
    step against the torch path of the same mpc.MPC call (torch evaluates and linearises the
    network, the kernels run the LinDx sweep)."""
    T, B = 10, 9
    net = _net(dilqr, ns, nc, hidden, "sigmoid", seed=ns + len(hidden)).to(dev)
    C_, c_, _, _, x0 = lindx_problem(ns, nc, T, B, torch.float64, seed=3)
    gm = dilqr.GradMethods.FINITE_DIFF if fd else dilqr.GradMethods.ANALYTIC

    def run():
        m = dilqr.MPC(ns, nc, T, u_lower=-1.0, u_upper=1.0, lqr_iter=1, verbose=-1,
                      exit_unconverged=False, detach_unconverged=False, grad_method=gm)
        with torch.no_grad():
            return m(x0.to(dev), dilqr.QuadCost(C_.to(dev), c_.to(dev)), net), m.last_info

    (x, u, costs), info = run()
    with monkeypatch.context() as mp:
        _torch_path(mp, dilqr)
        (xt, ut, ct), _ = run()
    assert rel(x, xt) < 1e-9 and rel(u, ut) < 1e-9 and rel(costs, ct) < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [[16], [10, 6]])
def test_gradients_7p3(dilqr, port, dev, monkeypatch, hidden):
    """mpc.MPC + NNDynamics on 7+3, boxed, with .backward(): every leaf against the torch path
    (both solves stop within eps of the fixed point: the tolerance of the NN golden tests), and
    dx0, dC, dc against port.kkt_backward at the runtime solution with F, f from the network
    there."""
    ns, nc, T, B = 7, 3, 10, 9
    kw = dict(u_lower=-1.0, u_upper=1.0)
    C_, c_, _, _, x0 = lindx_problem(ns, nc, T, B, torch.float64, seed=4)
    g = torch.Generator().manual_seed(12)
    gx = torch.randn(T, B, ns, generator=g, dtype=torch.float64)
    gu = torch.randn(T, B, nc, generator=g, dtype=torch.float64)

    def run():
        net = _net(dilqr, ns, nc, hidden, "sigmoid", seed=5).to(dev)
        leaves = [t.to(dev).requires_grad_() for t in (x0, C_, c_)]
        m = dilqr.MPC(ns, nc, T, lqr_iter=30, verbose=-1, exit_unconverged=False,
                      detach_unconverged=False, **kw)
        x, u, _ = m(leaves[0], dilqr.QuadCost(leaves[1], leaves[2]), net)
        ((x * gx.to(dev)).sum() + (u * gu.to(dev)).sum()).backward()
        grads = [t.grad for t in leaves] + [p.grad for fc in net.fcs for p in (fc.weight, fc.bias)]
        return x.detach(), u.detach(), grads, net, m.last_info

    x, u, grads, net, info = run()
    assert info._problem[0].dynamics == _lib().DYN_NN_RT
    with monkeypatch.context() as mp:
        _torch_path(mp, dilqr)
        _, _, grads_t, _, _ = run()
    for a, b in zip(grads, grads_t):
        assert rel(a, b) < 1e-6
    # the KKT problem at the runtime solution
    xs, us = x.cpu(), u.cpu()
    netc = net.cpu()
    _x, _u = xs[:-1].reshape(-1, ns), us[:-1].reshape(-1, nc)
    with torch.no_grad():
        nx = netc(_x, _u)
        R, S = netc.grad_input(_x, _u)
    f = (nx - torch.bmm(R, _x.unsqueeze(2)).squeeze(2) - torch.bmm(S, _u.unsqueeze(2)).squeeze(2))
    F = torch.cat((R, S), 2).reshape(T - 1, B, ns, ns + nc)
    k = port.kkt_backward(gx, gu, x0, C_, c_, F, f.reshape(T - 1, B, ns), xs, us, ns, nc, **kw)
    for mine, ref_, nm in zip(grads[:3], (k.dx_init, k.dC, k.dc), ("dx0", "dC", "dc")):
        assert rel(mine, ref_) < 1e-10, nm


@pytest.mark.gpu
def test_scale_7p3_solo2(sol, dilqr, dev):
    """7+3, one hidden layer of 32, boxed, T = 50, B = 65536 + 5, solo = 2: every problem is its
    own batch of one, so the first 64 problems of the full batch equal a B = 64 solve of them."""
    lib = _lib()
    ns, nc, T, B = 7, 3, 50, 65536 + 5
    net = _net(dilqr, ns, nc, [32], "sigmoid", seed=10)
    aux, ai = net._dilqr_pack(torch.float64, dev)
    dyn = sol.DynSpec(lib.DYN_NN, aux=aux, ai=ai)
    C_, c_, _, _, x0 = lindx_problem(ns, nc, T, 64, torch.float64, seed=10)
    reps = (B + 63) // 64
    g = torch.Generator(device=dev).manual_seed(13)
    Cb = C_.to(dev).repeat(1, reps, 1, 1)[:, :B].contiguous()
    cb = c_.to(dev).repeat(1, reps, 1)[:, :B].contiguous()
    cb[:, 64:] += torch.randn(cb[:, 64:].shape, generator=g, device=dev, dtype=cb.dtype)
    xb = x0.to(dev).repeat(reps, 1)[:B].contiguous()
    xb[64:] += torch.randn(xb[64:].shape, generator=g, device=dev, dtype=xb.dtype)
    kw = dict(u_lower=-1.0, u_upper=1.0, lqr_iter=10, verbose=-1, solo=2)
    X, U, Cst, info = sol.solve_mpc(xb, Cb, cb, dyn, ns, nc, T, **kw)
    torch.cuda.synchronize()
    assert info._problem[0].dynamics == lib.DYN_NN_RT
    x, u, cst, _ = sol.solve_mpc(xb[:64], Cb[:, :64], cb[:, :64], dyn, ns, nc, T, **kw)
    assert torch.isfinite(X).all() and torch.isfinite(U).all()
    assert rel(X[:, :64], x) <= 1e-12 and rel(U[:, :64], u) <= 1e-12 and rel(Cst[:64], cst) <= 1e-12
