"""Every solve option and the KKT gradients of every kernel family against the CPU oracle, in
FP64 and FP32, and results that do not depend on what ran earlier in the shared workspace.

Which kernels serve a call is not visible in it: `dilqr_lindx_kernels` / `dilqr_nn_kernels`
and `dilqr_mpc_plan` choose from the shape, the dtype, the bounds, `solo` and the batch.  Every
GPU case here asserts the family each of its solves ran (`info._problem[0].dynamics` and
`.group_sweep`, see `common.family`), so a change of plan fails the test instead of quietly
moving the coverage elsewhere.  The expected family comes from `common.expected_family`, a
table written out by hand, not from the library's rule.

Families:
  thread   one thread per problem (csrc/ilqr_kernels.cuh): compiled shapes whose per-warp
           stage fits, unless they are multi-input with batch-global bounds
  group    group sweep (csrc/group_kernels.cuh): compiled shapes too large to stage (FP64:
           6+2, 8+x, 13+3, 16+x; FP32: 8+4, 13+3, 16+x), and staged multi-input shapes with
           batch-global box constraints
  runtime  runtime-dimension LinDx kernels (csrc/rt_kernels.cuh): shapes without compiled kernels
  nn       compiled network kernels (NNDynamics 3+1, 4+2, 5+1)
  nn_rt    runtime-dimension network kernels

Shapes and the family of their solves ("box" = scalar or tensor bounds with solo = 0; the
KKT adjoint solve of Part 2 is always unbounded):

  shape     unbounded or solo   box             used in
            FP64     FP32       FP64    FP32
  1+1       runtime  runtime    runtime runtime 1
  4+2       thread   thread     group   group   1, 2
  5+1       thread   thread     thread  thread  1, 2, 3
  4+4       thread   thread     group   group   1
  6+2       group    thread     group   group   2
  8+2       group    thread     group   group   1
  8+4       group    group      group   group   1, 2, 3
  13+3      group    group      group   group   2
  16+4      group    group      group   group   1, 2
  7+3       runtime  runtime    runtime runtime 1, 2, 3
  24+8      runtime  runtime    runtime runtime 2
  31+1      runtime  runtime    runtime runtime 1
  NN 4+2    nn       nn         nn      nn      1, 2
  NN 6+2    nn_rt    nn_rt      nn_rt   nn_rt   1, 2

Part 1 (one teacher-forced LQR step against port.lqr_step in FP64 on the inputs as the device
gets them; x, u, costs, K, k within 3e-9 in FP64 and 3e-4 in FP32, the same line-search step,
the pnqp count exact in FP64) runs every option of
`OPTIONS` on every shape above in both dtypes, except: `chol_reg` needs n_ctrl > 1; the
networks take free, scalar box, pinned tensor box, u_zero_I, delta_u and solo.  So every
option meets every family in both dtypes.  Part 1b (CPU) checks that each option changes the
oracle's result by more than 100x the FP64 bound, so a device that ignored it would fail.

Part 2 (KKT gradients at the device's own solution against port.kkt_backward, through mpc.MPC
and LQRStep; 1e-10 in FP64, 1e-4 in FP32) runs free, scalar box, tensor box, no f and a
broadcast C[n,n] / c[n] on the shapes marked 2, both dtypes.  FP32 torch.ops.dilqr.lqr_kkt_backward
equals _solver.kkt_backward bitwise on one shape per family (5+1 thread, 8+4 group, 7+3 runtime).

Part 3 (workspace history, FP64): a solve after other solves on the same stream, warm-started
after a different problem of its shape, and interleaved forward / backward pairs through
mpc.MPC (5+1, 8+4, 7+3) and mpc_explicit.MPC (cartpole), against runs on a fresh workspace."""
import importlib
import math

import pytest
import torch

from common import (LINDX_COMPILED, NN_COMPILED, env_problem, expected_family, family,
                    lindx_problem, rel)

F64, F32 = torch.float64, torch.float32
STEP_TOL = {F64: 3e-9, F32: 3e-4}
KKT_TOL = {F64: 1e-10, F32: 1e-4}
T_STEP, T_KKT = 8, 10
BOX = 0.5                            # the scalar box [-BOX, BOX]


def _lib():
    return importlib.import_module("differentiable-ilqr_b200._lib")


# ------------------------------------------------------------------ problems
# (name, B, options).  Keys: bounds "scalar" / "tensor"; pin (some tensor bounds lo == hi);
# zero_I; delta_u; chol_reg (with the controls rescaled so that the 1e-6 I of the Cholesky
# solve moves the gains well beyond round-off); bcast 1 (C[T,n,n]) / 2 (C[n,n]); no_f; solo.
OPTIONS = [
    ("free", 33, dict()),
    ("scalar_box", 1, dict(bounds="scalar")),
    ("scalar_box_70", 70, dict(bounds="scalar")),
    ("tensor_box_pinned", 33, dict(bounds="tensor", pin=True)),
    ("u_zero_I", 70, dict(zero_I=True)),
    ("u_zero_I_box", 33, dict(zero_I=True, bounds="scalar")),
    ("delta_u_scalar", 33, dict(bounds="scalar", delta_u=0.3)),
    ("delta_u_tensor", 33, dict(bounds="tensor", delta_u=0.3)),
    ("chol_reg", 33, dict(chol_reg=True, ctrl_scale=0.1)),
    ("C_bcast1", 33, dict(bounds="scalar", bcast=1)),
    ("C_bcast2", 1, dict(bcast=2)),
    ("no_f", 33, dict(bounds="scalar", no_f=True)),
    ("solo1", 33, dict(bounds="tensor", delta_u=0.3, solo=1)),
]
# Per-problem pnqp flags change a result only when, in one pnqp iteration, a problem needs
# Armijo backtracking while another has already converged: the batch-global rule then stops
# backtracking after one pass.  Among the solo cases that happens on these shapes; on the
# others the solo case checks that per-problem flags leave the result right.
SOLO_MATTERS = {(8, 2), (16, 4)}
NN_OPTIONS = {"free", "scalar_box", "tensor_box_pinned", "u_zero_I", "delta_u_scalar", "solo1"}
# the option each case is about (Part 1b removes it and expects another result)
OPTION_KEY = {"scalar_box": "bounds", "scalar_box_70": "bounds", "tensor_box_pinned": "pin",
              "u_zero_I": "zero_I", "u_zero_I_box": "zero_I", "delta_u_scalar": "delta_u",
              "delta_u_tensor": "delta_u", "chol_reg": "chol_reg", "C_bcast1": "bcast",
              "C_bcast2": "bcast", "no_f": "no_f", "solo1": "solo"}

STEP_SHAPES = [(1, 1), (4, 2), (5, 1), (4, 4), (8, 2), (8, 4), (16, 4), (7, 3), (31, 1)]
NN_SHAPES = [(4, 2), (6, 2)]


def _box_global(opt):
    return opt.get("bounds") is not None and not opt.get("solo")


def _make(ns, nc, T, B, opt, seed):
    """FP64 inputs of one case: the LinDx problem, the bounds, the mask, the first iterate.
    Every random draw is taken whatever the options, so a case and the same case without one
    option (Part 1b) differ in that option only."""
    C_, c_, F, f, x0 = lindx_problem(ns, nc, T, B, F64, seed=seed)
    c_ = 3 * c_                      # unconstrained controls of a few units: the boxes bind
    g = torch.Generator().manual_seed(seed + 1)
    lo = -0.5 - torch.rand(T, B, nc, generator=g, dtype=F64)
    hi = 0.5 + torch.rand(T, B, nc, generator=g, dtype=F64)
    pinned = torch.rand(T, B, nc, generator=g) < 0.25
    v = torch.rand(T, B, nc, generator=g, dtype=F64) - 0.5
    zero_I = torch.rand(T, B, nc, generator=g) < 0.3
    u0 = 0.3 * torch.randn(T, B, nc, generator=g, dtype=F64)
    if opt.get("ctrl_scale"):
        # u = u'/s: Quu shrinks by s^2 (to about 1e-2), so the 1e-6 I of the Cholesky solve
        # moves the gains by about 1e-4 relative; the problem's conditioning is unchanged
        s = torch.ones(ns + nc, dtype=F64)
        s[ns:] = opt["ctrl_scale"]
        C_ = C_ * s[:, None] * s[None, :]
        c_ = c_ * s
        F = F * s
    kw = {}
    if opt.get("bounds") == "scalar":
        kw.update(u_lower=-BOX, u_upper=BOX)
    elif opt.get("bounds") == "tensor":
        if opt.get("pin"):           # lo == hi: x == lo and x == hi both hold inside pnqp
            lo, hi = torch.where(pinned, v, lo), torch.where(pinned, v, hi)
        kw.update(u_lower=lo, u_upper=hi)
    if opt.get("zero_I"):
        kw["u_zero_I"] = zero_I
    if "delta_u" in opt:
        kw["delta_u"] = opt["delta_u"]
    return dict(C=C_, c=c_, F=F, f=None if opt.get("no_f") else f, x0=x0, u0=u0, kw=kw)


def _to(p, dtype):
    q = {k: (v.to(dtype) if torch.is_tensor(v) and v.is_floating_point() else v)
         for k, v in p.items() if k != "kw"}
    q["kw"] = {k: (v.to(dtype) if torch.is_tensor(v) and v.is_floating_point() else v)
               for k, v in p["kw"].items()}
    return q


def _bcast(t, opt):
    """The cost tensor handed to the device for a broadcast option (C[T,n,n] or C[n,n])."""
    if opt.get("bcast") == 1:
        return t[:, 0].contiguous()
    if opt.get("bcast") == 2:
        return t[0, 0].contiguous()
    return t


def _dense(t, opt):
    """What the oracle gets for a broadcast option: the dense expansion of the broadcast base."""
    T, B = t.shape[0], t.shape[1]
    b = _bcast(t, opt)
    if opt.get("bcast") == 1:
        return b.unsqueeze(1).expand(T, B, *b.shape[1:]).contiguous()
    if opt.get("bcast") == 2:
        return b.expand(T, B, *b.shape).contiguous()
    return t


def _net_weights(ns, nc, seed, hidden=16):
    """One hidden layer, sigmoid, passthrough: (W1, b1, W2, b2) in FP64."""
    g = torch.Generator().manual_seed(seed)
    n = ns + nc
    W1 = torch.randn(hidden, n, generator=g, dtype=F64) / n ** 0.5
    b1 = 0.1 * torch.randn(hidden, generator=g, dtype=F64)
    W2 = 0.3 * torch.randn(ns, hidden, generator=g, dtype=F64) / hidden ** 0.5
    b2 = 0.1 * torch.randn(ns, generator=g, dtype=F64)
    return W1, b1, W2, b2


def _net_module(dilqr, ns, nc, W, dtype, dev):
    net = dilqr.NNDynamics(ns, nc, hidden_sizes=[W[0].shape[0]], activation="sigmoid",
                           passthrough=True).to(dtype)
    with torch.no_grad():
        for fc, (w, b) in zip(net.fcs, ((W[0], W[1]), (W[2], W[3]))):
            fc.weight.copy_(w)
            fc.bias.copy_(b)
    return net.to(dev)


def _select(p, b):
    """Problem b of a batch, as a batch of one."""
    def sel(v, dim):
        return v[:, b:b + 1] if dim else v[b:b + 1]
    q = dict(C=sel(p["C"], 1), c=sel(p["c"], 1), F=sel(p["F"], 1),
             f=None if p["f"] is None else sel(p["f"], 1), x0=sel(p["x0"], 0), u0=sel(p["u0"], 1))
    q["kw"] = {k: (sel(v, 1) if torch.is_tensor(v) else v) for k, v in p["kw"].items()}
    return q


def oracle_step(port, ns, nc, p, opt, W=None):
    """port.lqr_step on the case, teacher-forced at (x_cur, u0); per problem for solo."""
    T = p["C"].shape[0]
    if opt.get("solo"):
        outs = [oracle_step(port, ns, nc, _select(p, b), dict(opt, solo=0), W)
                for b in range(p["x0"].shape[0])]
        cat = lambda xs, d: torch.cat(xs, d)
        return dict(x=cat([o["x"] for o in outs], 1), u=cat([o["u"] for o in outs], 1),
                    costs=cat([o["costs"] for o in outs], 0), K=cat([o["K"] for o in outs], 1),
                    k=cat([o["k"] for o in outs], 1), alphas=cat([o["alphas"] for o in outs], 0),
                    n_qp=None, xc=cat([o["xc"] for o in outs], 1))
    Cd, cd = _dense(p["C"], opt), _dense(p["c"], opt)
    dt = p["x0"].dtype
    if W is None:
        dyn = port.LinDx(p["F"], p["f"])
        xc = port.get_traj(T, p["u0"], p["x0"], dyn)
        F = p["F"]
    else:
        dyn = port.NNDynamics(*(w.to(dt) for w in W), activation="sigmoid")
        xc = port.get_traj(T, p["u0"], p["x0"], dyn)
        F, _ = port.linearize_dynamics(xc, p["u0"], dyn)
    kw = dict(p["kw"])
    o = port.lqr_step(p["x0"], Cd, cd, F, xc, p["u0"], port.QuadCost(Cd, cd), dyn, ns, nc,
                      gain_solve="chol_reg" if opt.get("chol_reg") else "pinv", **kw)
    return dict(x=o.x, u=o.u, costs=o.costs, K=torch.stack(o.Ks[::-1]), k=torch.stack(o.ks[::-1]),
                alphas=o.alphas, n_qp=o.n_total_qp_iter, xc=xc)


def _step_cases():
    out = []
    for name, B, opt in OPTIONS:
        for ns, nc in STEP_SHAPES:
            if name == "chol_reg" and nc == 1:
                continue
            out.append(pytest.param(False, ns, nc, name, B, opt, id="%d+%d-%s" % (ns, nc, name)))
        if name in NN_OPTIONS:
            for ns, nc in NN_SHAPES:
                out.append(pytest.param(True, ns, nc, name, B, opt, id="nn%d+%d-%s" % (ns, nc, name)))
    return out


# ------------------------------------------------------------------ Part 1b (CPU)
@pytest.mark.parametrize("name,B,opt", [o for o in OPTIONS if o[0] in OPTION_KEY],
                         ids=[o[0] for o in OPTIONS if o[0] in OPTION_KEY])
def test_option_changes_oracle_result(port, name, B, opt):
    """Without its option a case computes something else, by more than 100x the FP64 bound of
    Part 1: a device that ignored the option could not pass Part 1.  Checked on every FP64
    case of Part 1 (same shapes, same seeds)."""
    key = OPTION_KEY[name]
    base = {k: v for k, v in opt.items() if k != key}
    for ns, nc in STEP_SHAPES:
        if (name == "chol_reg" and nc == 1) or (key == "solo" and (ns, nc) not in SOLO_MATTERS):
            continue
        seed = 100 + 7 * OPTIONS.index((name, B, opt)) + ns
        a = oracle_step(port, ns, nc, _make(ns, nc, T_STEP, B, opt, seed), opt)
        b = oracle_step(port, ns, nc, _make(ns, nc, T_STEP, B, base, seed), base)
        d = max(rel(a[k], b[k]) for k in ("x", "u", "K", "k"))
        assert d > 100 * STEP_TOL[F64], (name, ns, nc, d)
    if name in NN_OPTIONS and key != "solo":
        for ns, nc in NN_SHAPES:
            seed = 100 + 7 * OPTIONS.index((name, B, opt)) + ns
            W = _net_weights(ns, nc, seed=ns * 10 + nc)
            a = oracle_step(port, ns, nc, _make(ns, nc, T_STEP, B, opt, seed), opt, W)
            b = oracle_step(port, ns, nc, _make(ns, nc, T_STEP, B, base, seed), base, W)
            d = max(rel(a[k], b[k]) for k in ("x", "u", "K", "k"))
            assert d > 100 * STEP_TOL[F64], (name, "nn", ns, nc, d)


def test_family_table_matches_library():
    """The hand-written family table agrees with the library's choice of kernels (the plan's
    device-dependent part, the group sweep's batch capacity, is checked on the GPU)."""
    lib = _lib()
    L = lib.lib()
    for dt, dtype in ((lib.F64, F64), (lib.F32, F32)):
        for ns, nc in STEP_SHAPES + [(6, 2), (13, 3), (24, 8)]:
            want = lib.DYN_LINDX if (ns, nc) in LINDX_COMPILED else lib.DYN_LINDX_RT
            assert L.dilqr_lindx_kernels(dt, ns, nc) == want
        for ns, nc in NN_SHAPES:
            want = lib.DYN_NN if (ns, nc) in NN_COMPILED else lib.DYN_NN_RT
            assert L.dilqr_nn_kernels(dt, ns, nc) == want
    assert expected_family(6, 2, F64, False) == "group" and expected_family(6, 2, F32, False) == "thread"


# ------------------------------------------------------------------ GPU fixtures
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def sol():
    return importlib.import_module("differentiable-ilqr_b200._solver")


@pytest.fixture
def families(sol, monkeypatch):
    """The family of every solve_mpc call from here on (forward solves, the KKT adjoint solve)."""
    seen = []
    orig = sol.solve_mpc

    def recorded(*a, **kw):
        out = orig(*a, **kw)
        seen.append(family(out[3]))
        return out

    monkeypatch.setattr(sol, "solve_mpc", recorded)
    return seen


def fresh_stream(sol, dev):
    """A stream with no workspace yet.  torch hands streams out of a small pool, so a new
    Stream object may reuse a handle an earlier test solved on: drop its cached workspace."""
    s = torch.cuda.Stream(device=dev)
    sol._ws_cache.pop((dev.index if dev.index is not None else 0, s.cuda_stream), None)
    return s


def _on(dev, p):
    q = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in p.items() if k != "kw"}
    q["kw"] = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in p["kw"].items()}
    return q


# ------------------------------------------------------------------ Part 1 (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("nn,ns,nc,name,B,opt", _step_cases())
def test_step_option_vs_oracle(sol, port, dev, nn, ns, nc, name, B, opt, dtype):
    """One teacher-forced LQR step of each option on each family against port.lqr_step, run in
    FP64 on the inputs as the device gets them (rounded to `dtype`).  The oracle run in FP32
    is no reference: its pnqp can stall in FP32 where the kernels do not (see
    `_solo_problems_alone`)."""
    lib = _lib()
    seed = 100 + 7 * OPTIONS.index((name, B, opt)) + ns
    p = _to(_make(ns, nc, T_STEP, B, opt, seed), dtype)
    W = _net_weights(ns, nc, seed=ns * 10 + nc) if nn else None
    if nn:                       # the weights as the device gets them
        W = tuple(w.to(dtype).double() for w in W)
    o = oracle_step(port, ns, nc, _to(p, F64), opt, W)
    d = _on(dev, p)
    if nn:
        dilqr = importlib.import_module("differentiable-ilqr_b200")
        aux, ai = _net_module(dilqr, ns, nc, W, dtype, dev)._dilqr_pack(dtype, dev)
        dyn = sol.DynSpec(lib.DYN_NN, aux=aux, ai=ai)
    else:
        dyn = sol.DynSpec(lib.DYN_LINDX, F=d["F"], f=d["f"])
    x, u, costs, info = sol.solve_mpc(
        d["x0"], _bcast(d["C"], opt), _bcast(d["c"], opt), dyn, ns, nc, T_STEP,
        u_init=d["u0"], x_cur=o["xc"].to(dev), want_gains=True, verbose=-1,
        solo=opt.get("solo", 0), gain_solve=lib.GAIN_CHOL_REG if opt.get("chol_reg") else lib.GAIN_PLAIN,
        **d["kw"])
    assert family(info) == expected_family(ns, nc, dtype, _box_global(opt), nn)
    keep = torch.ones(B, dtype=torch.bool)
    if opt.get("solo"):
        keep = _solo_problems_alone(sol, dev, d, o, opt, dyn, ns, nc, (x, u, costs, info))
    tol = STEP_TOL[dtype]
    for k, v in (("x", x), ("u", u), ("costs", costs), ("K", info.K), ("k", info.k)):
        v, r = v.cpu(), o[k]
        if k == "costs":
            v, r = v[keep], r[keep]
        else:
            v, r = v[:, keep], r[:, keep]
        assert rel(v, r) < tol, (k, rel(v, r))
    # the same number of line-search decays (0.2 ** i) for every problem
    decays = lambda a: torch.round(torch.log(a.cpu().double()) / math.log(0.2))
    assert torch.equal(decays(info.alphas)[keep], decays(o["alphas"])[keep])
    if dtype == F64 and o["n_qp"] is not None:
        assert info.qp_iters[0] == o["n_qp"]


def _solo_problems_alone(sol, dev, d, o, opt, dyn, ns, nc, out):
    """Under solo = 1 every problem of the batch is a batch of one: its outputs equal, bit for
    bit, a solve of that problem alone.  Returns the problems to compare with the oracle: in
    FP32, those whose pnqp calls all converged.

    The others met the breakdown of the reference's pnqp in FP32 under per-problem Armijo
    flags.  Near the 1e-4 stop, a step of a little more than 1e-4 lowers the objective by less
    than the FP32 resolution of its value.  In the 4+4 case, a step of 1.6e-4 would lower an
    objective of a few units by 2e-7, below its FP32 spacing.  The Armijo ratio then comes out
    0, negative or NaN, the step is cut to 1e-10, and the search spends its 20 iterations at
    that point, 1.6e-4 from the solution.  Whether this happens depends on the last bits of
    the inputs: the oracle in FP32 meets it on other problems than the kernels do, and the
    oracle in FP64 does not meet it.  So no oracle predicts these problems' values.  For them
    the test checks the batch-of-one property, and that they are at most a tenth of the batch.
    Under batch-global flags a converged problem ends each Armijo loop after one pass, so the
    other cases do not meet it."""
    x, u, costs, info = out
    T, B = x.shape[0], x.shape[1]
    keep = torch.ones(B, dtype=torch.bool)
    lib = _lib()
    for b in range(B):
        one = lambda t, dim: None if t is None else (t[:, b:b + 1] if dim else t[b:b + 1])
        kw = {k: (one(v, 1) if torch.is_tensor(v) else v) for k, v in d["kw"].items()}
        dyn_b = dyn if dyn.kind != lib.DYN_LINDX else sol.DynSpec(
            lib.DYN_LINDX, F=one(d["F"], 1).contiguous(),
            f=None if d["f"] is None else one(d["f"], 1).contiguous())
        xb, ub, cb, ib = sol.solve_mpc(
            one(d["x0"], 0).contiguous(), _bcast(one(d["C"], 1).contiguous(), opt),
            _bcast(one(d["c"], 1).contiguous(), opt), dyn_b, ns, nc, T,
            u_init=one(d["u0"], 1).contiguous(), x_cur=one(o["xc"], 1).to(dev).contiguous(),
            want_gains=True, verbose=-1, solo=0, **kw)
        for mine, alone in ((x, xb), (u, ub), (info.K, ib.K), (info.k, ib.k)):
            assert torch.equal(mine[:, b:b + 1], alone), b
        assert torch.equal(costs[b:b + 1], cb) and torch.equal(info.alphas[b:b + 1], ib.alphas), b
        keep[b] = ib.pnqp_unconverged == 0
    if x.dtype == F64:           # no breakdown: every problem meets the oracle
        return torch.ones(B, dtype=torch.bool)
    assert int((~keep).sum()) * 10 <= B, int((~keep).sum())
    return keep


# ------------------------------------------------------------------ Part 2 (GPU)
KKT_SHAPES = [(4, 2), (5, 1), (6, 2), (8, 4), (13, 3), (16, 4), (7, 3), (24, 8)]
KKT_OPTIONS = [("free", dict()), ("scalar_box", dict(bounds="scalar")),
               ("tensor_box", dict(bounds="tensor")), ("no_f", dict(bounds="scalar", no_f=True)),
               ("C_bcast2", dict(bounds="scalar", bcast=2))]


def _kkt_oracle(port, ns, nc, p, opt, x, u, gx, gu, F=None, f=None):
    """port.kkt_backward in FP64 at the device's solution; the dense gradient of a broadcast
    cost summed over its broadcast axes."""
    up = lambda t: None if t is None else t.detach().cpu().double()
    kw = {k: (up(v) if torch.is_tensor(v) else v) for k, v in p["kw"].items()}
    Cd, cd = _dense(up(p["C"]), opt), _dense(up(p["c"]), opt)
    if F is None:                       # LinDx: the problem's own dynamics
        F, f = up(p["F"]), up(p["f"])
    k = port.kkt_backward(up(gx), up(gu), up(p["x0"]), Cd, cd, F, f, up(x), up(u), ns, nc, **kw)
    dC, dc = k.dC, k.dc
    if opt.get("bcast") == 2:
        dC, dc = dC.sum((0, 1)), dc.sum((0, 1))
    return k._replace(dC=dC, dc=dc)


def _active(u, kw):
    lo, hi = kw["u_lower"], kw["u_upper"]
    return (torch.abs(u - lo) <= 1e-8) | (torch.abs(u - hi) <= 1e-8)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("entry", ["mpc", "lqr_step"])
@pytest.mark.parametrize("name,opt", KKT_OPTIONS, ids=[o[0] for o in KKT_OPTIONS])
@pytest.mark.parametrize("ns,nc", KKT_SHAPES, ids=["%d+%d" % s for s in KKT_SHAPES])
def test_kkt_gradients_vs_oracle(sol, port, dev, families, ns, nc, name, opt, entry, dtype):
    """dx0, dC, dc, dF, df of mpc.MPC / LQRStep against port.kkt_backward at the device's own
    (x, u), every input upcast to FP64: what is left is the backward's own round-off."""
    dilqr = importlib.import_module("differentiable-ilqr_b200")
    B = 9 if ns + nc > 16 else 33
    p = _to(_make(ns, nc, T_KKT, B, opt, seed=300 + ns + nc), dtype)
    d = _on(dev, p)
    Cl = _bcast(d["C"], opt).clone().requires_grad_()
    cl = _bcast(d["c"], opt).clone().requires_grad_()
    leaves = [d["x0"].clone().requires_grad_(), Cl, cl, d["F"].clone().requires_grad_()]
    if d["f"] is not None:
        leaves.append(d["f"].clone().requires_grad_())
    f_in = leaves[4] if d["f"] is not None else None
    n = ns + nc
    if entry == "mpc":
        m = dilqr.MPC(ns, nc, T_KKT, lqr_iter=20, verbose=-1, exit_unconverged=False,
                      detach_unconverged=False, n_batch=B, **d["kw"])
        x, u, _ = m(leaves[0], dilqr.QuadCost(Cl, cl), dilqr.LinDx(leaves[3], f_in))
    else:
        xc = port.get_traj(T_KKT, p["u0"], p["x0"], port.LinDx(p["F"], p["f"])).to(dev)
        Ce = Cl.expand(T_KKT, B, n, n) if opt.get("bcast") else Cl
        ce = cl.expand(T_KKT, B, n) if opt.get("bcast") else cl
        step = dilqr.LQRStep(ns, nc, T_KKT, current_x=xc, current_u=d["u0"], **d["kw"])
        x, u = step(leaves[0], Ce, ce, leaves[3], f_in)[:2]
    g = torch.Generator().manual_seed(12)
    gx = torch.randn(x.shape, generator=g, dtype=F64).to(dtype)
    gu = torch.randn(u.shape, generator=g, dtype=F64).to(dtype)
    ((x * gx.to(dev)).sum() + (u * gu.to(dev)).sum()).backward()
    box = opt.get("bounds") is not None
    assert families == [expected_family(ns, nc, dtype, box), expected_family(ns, nc, dtype, False)]
    if box:
        assert bool(_active(u.detach(), d["kw"]).any())
    k = _kkt_oracle(port, ns, nc, p, opt, x, u, gx, gu)
    refs = [k.dx_init, k.dC, k.dc, k.dF] + ([k.df] if d["f"] is not None else [])
    for i, (leaf, r) in enumerate(zip(leaves, refs)):
        assert rel(leaf.grad, r) < KKT_TOL[dtype], (("dx0", "dC", "dc", "dF", "df")[i], rel(leaf.grad, r))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("name,opt", [o for o in KKT_OPTIONS if o[0] != "no_f"],
                         ids=[o[0] for o in KKT_OPTIONS if o[0] != "no_f"])
@pytest.mark.parametrize("ns,nc", NN_SHAPES, ids=["nn%d+%d" % s for s in NN_SHAPES])
def test_network_kkt_gradients_vs_oracle(sol, port, dev, families, ns, nc, name, opt, dtype):
    """mpc.MPC with NNDynamics: dx0, dC, dc against port.kkt_backward at the device's solution
    with F, f the network's linearisation there (FP64, from the upcast solution)."""
    dilqr = importlib.import_module("differentiable-ilqr_b200")
    T, B = T_KKT, 33
    p = _to(_make(ns, nc, T, B, opt, seed=400 + ns), dtype)
    d = _on(dev, p)
    W = _net_weights(ns, nc, seed=ns * 10 + nc)
    net = _net_module(dilqr, ns, nc, W, dtype, dev)
    Cl = _bcast(d["C"], opt).clone().requires_grad_()
    cl = _bcast(d["c"], opt).clone().requires_grad_()
    x0 = d["x0"].clone().requires_grad_()
    m = dilqr.MPC(ns, nc, T, lqr_iter=20, verbose=-1, exit_unconverged=False,
                  detach_unconverged=False, n_batch=B, **d["kw"])
    x, u, _ = m(x0, dilqr.QuadCost(Cl, cl), net)
    g = torch.Generator().manual_seed(12)
    gx = torch.randn(x.shape, generator=g, dtype=F64).to(dtype)
    gu = torch.randn(u.shape, generator=g, dtype=F64).to(dtype)
    ((x * gx.to(dev)).sum() + (u * gu.to(dev)).sum()).backward()
    box = opt.get("bounds") is not None
    assert families == [expected_family(ns, nc, dtype, box, nn=True),
                        expected_family(ns, nc, dtype, False)]
    if box:
        assert bool(_active(u.detach(), d["kw"]).any())
    xs, us = x.detach().cpu().double(), u.detach().cpu().double()
    on = port.NNDynamics(*W, activation="sigmoid")
    F, fv = port.linearize_dynamics(xs, us, on)
    k = _kkt_oracle(port, ns, nc, p, opt, x, u, gx, gu, F=F, f=fv)
    for leaf, r, nm in zip((x0, Cl, cl), (k.dx_init, k.dC, k.dc), ("dx0", "dC", "dc")):
        assert rel(leaf.grad, r) < KKT_TOL[dtype], (nm, rel(leaf.grad, r))


@pytest.mark.gpu
@pytest.mark.parametrize("ns,nc,fam", [(5, 1, "thread"), (8, 4, "group"), (7, 3, "runtime")])
def test_torch_op_kkt_backward_f32(sol, dev, families, ns, nc, fam):
    """FP32 torch.ops.dilqr.lqr_kkt_backward is bitwise _solver.kkt_backward."""
    ops = importlib.import_module("differentiable-ilqr_b200.torch_ops")
    ops.load()
    lib = _lib()
    T, B = T_KKT, 33
    p = _on(dev, _to(_make(ns, nc, T, B, dict(bounds="scalar"), seed=500 + ns), F32))
    x, u, _, info = sol.solve_mpc(p["x0"], p["C"], p["c"], sol.DynSpec(lib.DYN_LINDX, F=p["F"], f=p["f"]),
                                  ns, nc, T, u_lower=-BOX, u_upper=BOX, lqr_iter=10, verbose=-1)
    assert bool(_active(u, dict(u_lower=-BOX, u_upper=BOX)).any())
    g = torch.Generator().manual_seed(9)
    gx = torch.randn(T, B, ns, generator=g).to(dev)
    gu = torch.randn(T, B, nc, generator=g).to(dev)
    a = torch.ops.dilqr.lqr_kkt_backward(gx, gu, p["x0"], p["C"], p["c"], p["F"], x, u, -BOX, BOX)
    b = sol.kkt_backward(gx, gu, p["x0"], p["C"], p["c"], p["F"], p["f"], x, u, ns, nc,
                         u_lower=-BOX, u_upper=BOX)
    assert families[-1] == fam == expected_family(ns, nc, F32, False)
    for ta, tb, nm in zip(a, b, ("dx0", "dC", "dc", "dF", "df")):
        assert ta.dtype == F32 and torch.equal(ta, tb), nm


# ------------------------------------------------------------------ Part 3 (GPU)
def _solve10(sol, dev, ns, nc, seed, bounds="scalar", solo=0, u_init=False, B=33):
    lib = _lib()
    p = _on(dev, _make(ns, nc, T_STEP, B, dict(bounds=bounds), seed))
    kw = dict(p["kw"])
    if u_init:
        kw["u_init"] = p["u0"]
    return sol.solve_mpc(p["x0"], p["C"], p["c"], sol.DynSpec(lib.DYN_LINDX, F=p["F"], f=p["f"]),
                         ns, nc, T_STEP, lqr_iter=10, verbose=-1, solo=solo, **kw)


def _same_solve(a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    assert a[3].qp_iters == b[3].qp_iters and a[3].n_iters == b[3].n_iters


@pytest.mark.gpu
@pytest.mark.parametrize("ns,nc,fam", [(5, 1, "thread"), (8, 4, "group"), (7, 3, "runtime")])
def test_solve_independent_of_earlier_solves(sol, dev, ns, nc, fam):
    """A boxed, batch-global 10-iteration solve after solves of another shape, another bounds
    kind and solo = 1 on the same stream, and warm-started after a different problem of its
    own shape (so the carried pnqp trace guess is wrong), equals the solve on a fresh
    workspace bitwise, per-iteration pnqp counts included."""
    with torch.cuda.stream(fresh_stream(sol, dev)):
        ref = _solve10(sol, dev, ns, nc, seed=1)
        torch.cuda.current_stream().synchronize()
    with torch.cuda.stream(fresh_stream(sol, dev)):
        ref_warm_fresh = _solve10(sol, dev, ns, nc, seed=1, u_init=True)
        torch.cuda.current_stream().synchronize()
    assert family(ref[3]) == fam == expected_family(ns, nc, F64, True)
    assert not ref_warm_fresh[3]._problem[0].keep_trace_guess
    with torch.cuda.stream(fresh_stream(sol, dev)):
        _solve10(sol, dev, 4, 2, seed=2, bounds=None)
        _solve10(sol, dev, 16, 4, seed=3, B=70)
        _solve10(sol, dev, ns, nc, seed=4, bounds="tensor")
        _solve10(sol, dev, ns, nc, seed=5, solo=1)
        after = _solve10(sol, dev, ns, nc, seed=1)
        _solve10(sol, dev, ns, nc, seed=6, u_init=True)
        warm = _solve10(sol, dev, ns, nc, seed=1, u_init=True)
        torch.cuda.current_stream().synchronize()
    _same_solve(after, ref)
    assert warm[3]._problem[0].keep_trace_guess == 1
    _same_solve(warm, ref_warm_fresh)


def _mpc_grads(dilqr, dev, ns, nc, seed):
    """Forward of one boxed LinDx problem through mpc.MPC; returns (x, u, a backward closure)."""
    p = _on(dev, _make(ns, nc, T_KKT, 33, dict(bounds="scalar"), seed))
    leaves = [p[k].clone().requires_grad_() for k in ("x0", "C", "c", "F", "f")]
    m = dilqr.MPC(ns, nc, T_KKT, lqr_iter=20, verbose=-1, exit_unconverged=False,
                  detach_unconverged=False, u_lower=-BOX, u_upper=BOX)
    x, u, _ = m(leaves[0], dilqr.QuadCost(leaves[1], leaves[2]), dilqr.LinDx(leaves[3], leaves[4]))
    g = torch.Generator().manual_seed(seed)
    gx = torch.randn(x.shape, generator=g, dtype=F64).to(dev)
    gu = torch.randn(u.shape, generator=g, dtype=F64).to(dev)

    def backward():
        ((x * gx).sum() + (u * gu).sum()).backward()
        return [t.grad for t in leaves]
    return x.detach(), u.detach(), backward


@pytest.mark.gpu
@pytest.mark.parametrize("ns,nc", [(5, 1), (8, 4), (7, 3)])
def test_interleaved_lindx_backward(sol, dev, ns, nc):
    """forward A, forward B, backward B, backward A on one stream through mpc.MPC: the
    gradients equal those of A and B solved and differentiated alone, bitwise."""
    dilqr = importlib.import_module("differentiable-ilqr_b200")
    alone = []
    for seed in (1, 2):
        with torch.cuda.stream(fresh_stream(sol, dev)):
            xa, ua, bwd = _mpc_grads(dilqr, dev, ns, nc, seed)
            alone.append((xa, ua, bwd()))
            torch.cuda.current_stream().synchronize()
    with torch.cuda.stream(fresh_stream(sol, dev)):
        xa, ua, bwd_a = _mpc_grads(dilqr, dev, ns, nc, 1)
        xb, ub, bwd_b = _mpc_grads(dilqr, dev, ns, nc, 2)
        gb = bwd_b()
        ga = bwd_a()
        torch.cuda.current_stream().synchronize()
    for (x0, u0, g0), (x1, u1, g1) in zip(alone, ((xa, ua, ga), (xb, ub, gb))):
        assert torch.equal(x0, x1) and torch.equal(u0, u1)
        for a, b, nm in zip(g0, g1, ("dx0", "dC", "dc", "dF", "df")):
            assert torch.equal(a, b), nm


@pytest.mark.gpu
def test_interleaved_dilqr_backward(sol, port, dev, monkeypatch):
    """forward A, forward B, backward B, backward A through mpc_explicit.MPC (cartpole, fused
    DiLQR backward).  B's solve reused the workspace A's fused preparation reads (gains, packed
    C), so ws.gen sends A's backward back through dilqr_prepare; its gradients match A's alone
    to 1e-12 (the bound by which the fused and round-1 sequences agree), B's are bitwise."""
    dilqr = importlib.import_module("differentiable-ilqr_b200")
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    calls = []
    orig = sol.dilqr_prepare

    def counted(*a, **kw):
        calls.append(kw.get("solve_info") is not None)
        return orig(*a, **kw)

    monkeypatch.setattr(sol, "dilqr_prepare", counted)
    T, B = 20, 33

    def forward(seed):
        pdx, x0, C, c, kw = env_problem(port, "cartpole", T, B, F64, sigma=0.2, seed=seed)
        kw["eps"] = 1e-9
        theta = pdx.params.to(dev).requires_grad_()
        Cg, cg = C.to(dev).requires_grad_(), c.to(dev).requires_grad_()
        m = dilqr.mpc_explicit.MPC(5, 1, T, lqr_iter=30, verbose=-1, exit_unconverged=False,
                                   detach_unconverged=False, richardson_passes=40,
                                   richardson_tol=None, **kw)
        x, u, _ = m(x0.to(dev), dilqr.QuadCost(Cg, cg), env.CartpoleDx(theta))
        g = torch.Generator().manual_seed(seed)
        gx = torch.randn(x.shape, generator=g, dtype=F64).to(dev)
        gu = torch.randn(u.shape, generator=g, dtype=F64).to(dev)

        def backward():
            ((x * gx).sum() + (u * gu).sum()).backward()
            return m.last_backward["fused"], [theta.grad, Cg.grad, cg.grad]
        return x.detach(), u.detach(), backward

    alone = []
    for seed in (1, 2):
        with torch.cuda.stream(fresh_stream(sol, dev)):
            x, u, bwd = forward(seed)
            alone.append((x, u) + bwd())
            torch.cuda.current_stream().synchronize()
    assert alone[0][2] and alone[1][2]          # alone, both run the fused backward
    del calls[:]
    with torch.cuda.stream(fresh_stream(sol, dev)):
        xa, ua, bwd_a = forward(1)
        xb, ub, bwd_b = forward(2)
        fused_b, gb = bwd_b()
        fused_a, ga = bwd_a()
        torch.cuda.current_stream().synchronize()
    # the two forwards, then A's backward prepares again, without the (stale) solve
    assert calls == [True, True, False]
    assert fused_b and not fused_a
    assert torch.equal(xa, alone[0][0]) and torch.equal(ua, alone[0][1])
    assert torch.equal(xb, alone[1][0]) and torch.equal(ub, alone[1][1])
    for a, b in zip(ga, alone[0][3]):
        assert rel(a, b) < 1e-12, rel(a, b)
    for a, b in zip(gb, alone[1][3]):
        assert torch.equal(a, b)
