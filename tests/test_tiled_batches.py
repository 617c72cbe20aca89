"""Every kernel family at production batch sizes: a tiled batch reproduces its base bit for bit.

The oracle tests run at B <= ~130, where a solve launches one to three blocks.  Users (and
bench.py) run B = 65536 per GPU, where other code runs: commit kernels of hundreds of blocks
folded by the block that takes the last ticket, the group sweep's batch loop and its phase-B
barrier over many blocks, trace replay past the group sweep's capacity, per-warp partials of
the backward's reductions, and offsets past 2^31 elements.  The oracle cannot be run at that
size, and it is not invariant to the batch size in the last bit anyway (torch sums over the
batch, and the line search compares costs that tie to the last bit).  The device is: each
problem's arithmetic is the same wherever the problem sits.

The check: take a base of K distinct problems and build a batch of B where problem b is base
problem b % K (every per-problem tensor: x_init, C, c, F, f, tensor bounds, u_zero_I, expert
controls, upstream gradients).  Every batch-global decision of the algorithm (pnqp's exit and
Armijo loop, the line-search loop, the not-improved rule, the pnqp count) is a function of the
*set* of distinct problems, so the tiled batch makes the decisions of its base, and every copy
of base problem j must equal, bit for bit, what the device returns for j in a solve of the base
alone.  K = 41 is an odd prime and no B below is a multiple of it: a problem read from warp
+-1, block +-1 or group +-1 lands on another base problem, and the last copy is partial.  (Not
37: the B200 has 148 = 4 * 37 SMs, so the group sweep's capacity is a multiple of 37.)

Kept out: `full_du_norm` (its rows mix problems, lqr_step.py:243-245), so `du` is not compared
and `detach_unconverged=False`; the eps stop rule (not invariant either): eps = 0 and every
solve asserts n_iters == lqr_iter.

Batch sums (a broadcast cost's gradient, dtheta, the imitation step's outputs) are compared
with sum_j m_j g_j, m_j the number of copies of j and g_j the base's per-problem value, within
tol * sum_j m_j |g_j| (1e-12 FP64, 1e-5 FP32).

Every GPU case asserts the family of its solves (common.expected_family) and, for the group
sweep, that its B is in the intended regime: within one pass of the groups, looping over the
batch (ceil(B / 16) groups > cap / 256 blocks), or past the capacity (trace replay).  The
capacity comes from dilqr_mpc_plan on the device (`group_capacity`).  There the family
changes, so at cap + 1 copies are compared among themselves bitwise and with the base within
1e-9 (FP64) / 1e-4 (FP32) with exact pnqp counts, as test_rocket_full_size_group_sweep_properties
does at full size.

Each base is checked against the oracle by `test_base_vs_oracle` (end to end, 1e-6, exact pnqp
counts, FP64 as test_env_vs_oracle), `test_kkt_tiled` (port.kkt_backward at the device's own
solution, 1e-10 as test_kkt_gradients_vs_oracle) and `test_pnqp_tiled` (port.pnqp as
test_pnqp_standalone).  The DiLQR bases (cartpole scalar box, pendulum tensor bounds, tiled
cost) are the configurations of test_dilqr_backward_paths (fused-cartpole-dense,
generic-pendulum-bounds, fused-cartpole-tile) at another horizon and batch."""
import ctypes
import importlib
import time

import pytest
import torch

from common import env_problem, expected_family, family, lindx_problem, rel

F64, F32 = torch.float64, torch.float32
K = 41                               # base problems: an odd prime, no B below is a multiple
B_FULL = 65541                       # 2^16 + 5
SUM_TOL = {F64: 1e-12, F32: 1e-5}
BOX = 0.5
GROUP_LANES, GROUP_THREADS = 16, 256  # group_kernels.cuh: G lanes per problem (n <= 16), block


def _lib():
    return importlib.import_module("differentiable-ilqr_b200._lib")


# ------------------------------------------------------------------ helpers
def tile(t, dim, B, k):
    """Problem b of the result is problem b % k of ``t`` along ``dim`` (on t's device)."""
    return t.index_select(dim, torch.arange(B, device=t.device) % k)


def first_mismatch(big, base, k, dim):
    """None if every copy of ``big`` along ``dim`` equals its base problem bit for bit (the
    partial last copy included), else the first problem b that differs."""
    want = tile(base.to(big.device), dim, big.shape[dim], k)
    if big.shape == want.shape and big.dtype == want.dtype and torch.equal(big, want):
        return None
    if big.shape != want.shape:
        return 0
    ne = (big != want) | (torch.isnan(big) != torch.isnan(want))
    ne = ne.movedim(dim, 0).reshape(big.shape[dim], -1).any(1)
    return int(ne.nonzero()[0]) if bool(ne.any()) else None


def copies_equal(big, base, k, dim, what=""):
    b = first_mismatch(big, base, k, dim)
    assert b is None, ("%s: problem %d (copy of base problem %d) differs from its base: warp %d, "
                       "block of 128 %d, block of 256 %d" % (what, b, b % k, b // 32, b // 128, b // 256))


def copy_counts(B, k):
    return torch.bincount(torch.arange(B) % k, minlength=k)


def assert_batch_sum(got, per_problem, m, tol, what=""):
    """got = sum_j m_j g_j (g_j = per_problem[j]) within tol * sum_j m_j |g_j|, elementwise."""
    g = per_problem.detach().cpu().double()
    mw = m.double().reshape(-1, *([1] * (g.dim() - 1)))
    want, scale = (mw * g).sum(0), (mw * g.abs()).sum(0)
    err = (got.detach().cpu().double().reshape(want.shape) - want).abs()
    assert bool((err <= tol * scale).all()), (what, float((err / (scale + 1e-300)).max()))


def group_capacity(ns, nc, dyn, dtype):
    """The largest batch dilqr_mpc_plan gives the group sweep (a boxed, batch-global solve), by
    bisection on a bare DilqrSolve: planning allocates nothing."""
    lib = _lib()
    L = lib.lib()

    def group(B):
        s = lib.DilqrSolve()
        s.n_state, s.n_ctrl, s.T, s.n_batch = ns, nc, 10, B
        s.dtype, s.dynamics = (lib.F64 if dtype == F64 else lib.F32), dyn
        s.bounds_kind, s.solo = lib.BOUNDS_SCALAR, 0
        assert L.dilqr_mpc_plan(ctypes.byref(s)) == 0
        return s.group_sweep == 1
    lo, hi = 1, 1 << 26
    assert group(lo) and not group(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if group(mid) else (lo, mid)
    assert lo % GROUP_THREADS == 0, lo       # whole co-resident blocks of one thread per problem
    return lo


def need_memory(nbytes, what):
    """Skip, with the reason, when the device has less free memory than the case needs."""
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip("%s needs ~%.1f GB of device memory, %.1f GB free" % (what, nbytes / 1e9, free / 1e9))


def solve_bytes(B, T, ns, nc, dtype):
    """An upper estimate of a tiled solve's footprint from its shapes: the tiled inputs (C, c,
    F, f), the solver's copies (packed C, trajectories, gains, line-search state) and the
    outputs, with the base solve's outputs and the comparisons' temporaries."""
    n = ns + nc
    s = 4 if dtype == F32 else 8
    return int(1.2 * s * B * T * (2.5 * n * n + 2 * ns * n + 12 * n + 2 * nc * ns)) + (1 << 28)


@pytest.fixture(autouse=True)
def _report(request):
    """Wall time and peak device memory of every GPU case (printed; pytest -s shows them)."""
    gpu = request.node.get_closest_marker("gpu") is not None and torch.cuda.is_available()
    if gpu:
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    if gpu:
        torch.cuda.synchronize()
        print("\n[tiled] %s wall %.1f s peak %.2f GB" % (
            request.node.name, time.time() - t0, torch.cuda.max_memory_allocated() / 1e9))


# ------------------------------------------------------------------ cases
# name -> case.  env: the env_dx model (model box; rocket +-20); else LinDx (ns, nc) or, with
# nn, NNDynamics.  bounds: "scalar" (+-BOX) / "tensor" (per problem, with u_zero_I and a
# broadcast C[T,n,n]).  Bs: the batches; "cap" is the group sweep's capacity.
CASES = {
    "cartpole": dict(env="cartpole", ns=5, nc=1, T=50, L=10, Bs=[65536, B_FULL]),
    "pendulum": dict(env="pendulum", ns=3, nc=1, T=20, L=10, Bs=[B_FULL]),
    "rocket": dict(env="rocket", ns=13, nc=3, T=20, L=4, Bs=["cap", "cap+1"], dtypes=[F64]),
    "lindx5+1-box": dict(ns=5, nc=1, T=10, L=10, bounds="scalar", Bs=[B_FULL]),
    "lindx5+1-tensor": dict(ns=5, nc=1, T=10, L=10, bounds="tensor", Bs=[B_FULL]),
    "lindx4+2-free": dict(ns=4, nc=2, T=10, L=10, Bs=[B_FULL]),
    "lindx4+2-box": dict(ns=4, nc=2, T=10, L=10, bounds="scalar", Bs=[257, "cap/16+1", "cap"]),
    "lindx8+4-box": dict(ns=8, nc=4, T=10, L=10, bounds="scalar",
                         Bs=[257, "cap/16+1", "cap", "cap+1"]),
    "lindx7+3-box": dict(ns=7, nc=3, T=20, L=10, bounds="scalar", Bs=[B_FULL]),
    "lindx31+1-box": dict(ns=31, nc=1, T=10, L=10, bounds="scalar", Bs=[8197]),
    "nn4+2-box": dict(nn=True, ns=4, nc=2, T=10, L=10, bounds="scalar", Bs=[B_FULL]),
    "nn6+2-box": dict(nn=True, ns=6, nc=2, T=10, L=10, bounds="scalar", Bs=[B_FULL]),
    # C has 200 * 300007 * 36 > 2^31 elements: 64-bit offsets
    "lindx4+2-T200": dict(ns=4, nc=2, T=200, L=2, Bs=[300007], dtypes=[F32]),
}
BOXED = [n for n, c in CASES.items() if c.get("env") or c.get("bounds")]


def _net_weights(ns, nc, seed, hidden=16):
    g = torch.Generator().manual_seed(seed)
    n = ns + nc
    W1 = torch.randn(hidden, n, generator=g, dtype=F64) / n ** 0.5
    b1 = 0.1 * torch.randn(hidden, generator=g, dtype=F64)
    W2 = 0.3 * torch.randn(ns, hidden, generator=g, dtype=F64) / hidden ** 0.5
    b2 = 0.1 * torch.randn(ns, generator=g, dtype=F64)
    return W1, b1, W2, b2


def base_problem(port, name, k=K, seed=0):
    """The FP64 CPU inputs of k base problems.  Returns (problem, oracle dynamics, env model or
    None); problem keys: x0, C, c (dense [T,k,..] or shared), F, f, kw (solver keywords: bounds,
    u_zero_I, line search), W (network weights)."""
    c = CASES[name]
    T, ns, nc = c["T"], c["ns"], c["nc"]
    if c.get("env"):
        pdx, x0, C, cv, kw = env_problem(port, c["env"], T, k, F64, sigma=0.5, seed=seed)
        if c["env"] == "cartpole":      # bench.make_inputs (sigma = 0.5)
            bench = importlib.import_module("bench")
            x0 = bench.make_inputs(torch, k, F64, seed)[0]
        if c["env"] == "rocket":
            kw.update(u_lower=-20.0, u_upper=20.0)
        kw["eps"] = 0.0
        return dict(x0=x0, C=C, c=cv, F=None, f=None, kw=kw, W=None), pdx, pdx
    C, cv, F, f, x0 = lindx_problem(ns, nc, T, k, F64, seed=seed)
    cv = 3 * cv                          # unconstrained controls of a few units: the boxes bind
    kw = dict(eps=0.0)
    g = torch.Generator().manual_seed(seed + 1)
    if c.get("bounds") == "scalar":
        kw.update(u_lower=-BOX, u_upper=BOX)
    elif c.get("bounds") == "tensor":
        kw.update(u_lower=-0.2 - torch.rand(T, k, nc, generator=g, dtype=F64),
                  u_upper=0.2 + torch.rand(T, k, nc, generator=g, dtype=F64),
                  u_zero_I=torch.rand(T, k, nc, generator=g) < 0.3)
        C = C[:, 0].contiguous()         # C[T,n,n], shared by every problem
    W = None
    if c.get("nn"):
        W = _net_weights(ns, nc, seed=ns * 10 + nc)
        dyn = port.NNDynamics(*W, activation="sigmoid")
        F = f = None
    else:
        dyn = port.LinDx(F, f)
    return dict(x0=x0, C=C, c=cv, F=F, f=f, kw=kw, W=W), dyn, None


def _per_problem(name, key, t):
    """The batch dim of input ``key`` (None: shared by every problem)."""
    if t is None or not torch.is_tensor(t):
        return None
    if key == "x0":
        return 0
    if key == "C" and CASES[name].get("bounds") == "tensor":
        return None
    return 1


def _dense_C(C, T, k):
    return C[:, None].expand(T, k, *C.shape[1:]).contiguous() if C.dim() == 3 else C


def on_device(name, P, dtype, dev, B=None, k=K):
    """The problem in ``dtype`` on the device, tiled to B problems (B None: the base)."""
    def mv(key, t):
        if not torch.is_tensor(t):
            return t
        t = t.to(dev) if t.dtype == torch.bool else t.to(dev, dtype)
        d = _per_problem(name, key, t)
        return t.contiguous() if B is None or d is None else tile(t, d, B, k).contiguous()
    q = {key: mv(key, v) for key, v in P.items() if key not in ("kw", "W")}
    q["kw"] = {key: mv(key, v) for key, v in P["kw"].items()}
    q["W"] = P["W"]
    return q


def dyn_spec(sol, dilqr, name, d, dtype, dev, pdx):
    lib = _lib()
    c = CASES[name]
    if c.get("env"):
        env = importlib.import_module("differentiable-ilqr_b200.env_dx")
        cls = {"cartpole": env.CartpoleDx, "pendulum": env.PendulumDx, "rocket": env.RocketDx}[c["env"]]
        mpc = importlib.import_module("differentiable-ilqr_b200.mpc")
        return mpc._dyn_spec(cls(pdx.params.to(dev, dtype)))
    if c.get("nn"):
        net = dilqr.NNDynamics(c["ns"], c["nc"], hidden_sizes=[16], activation="sigmoid",
                               passthrough=True).to(dtype)
        with torch.no_grad():
            for fc, (w, b) in zip(net.fcs, ((d["W"][0], d["W"][1]), (d["W"][2], d["W"][3]))):
                fc.weight.copy_(w)
                fc.bias.copy_(b)
        aux, ai = net.to(dev)._dilqr_pack(dtype, dev)
        return sol.DynSpec(lib.DYN_NN, aux=aux, ai=ai)
    return sol.DynSpec(lib.DYN_LINDX, F=d["F"], f=d["f"])


def solve(sol, dilqr, name, d, dtype, dev, pdx):
    c = CASES[name]
    out = sol.solve_mpc(d["x0"], d["C"], d["c"], dyn_spec(sol, dilqr, name, d, dtype, dev, pdx),
                        c["ns"], c["nc"], c["T"], lqr_iter=c["L"], verbose=-1, want_gains=True,
                        **d["kw"])
    assert out[3].n_iters == c["L"]
    return out


def family_of(name, dtype, B, cap):
    c = CASES[name]
    if cap is not None and B > cap:
        return "thread"                  # trace replay
    if c.get("env"):
        return "group" if c["env"] == "rocket" else "thread"
    return expected_family(c["ns"], c["nc"], dtype, c.get("bounds") is not None, c.get("nn", False))


def resolve_B(spec, cap):
    if not isinstance(spec, str):
        return spec
    return {"cap": cap, "cap+1": cap + 1, "cap/16+1": cap // GROUP_LANES + 1}[spec]


def _fwd_params():
    out = []
    for name, c in CASES.items():
        for dtype in c.get("dtypes", [F64, F32]):
            for Bs in c["Bs"]:
                out.append(pytest.param(name, dtype, Bs, id="%s-%s-%s" % (
                    name, "f64" if dtype == F64 else "f32", Bs)))
    return out


# ------------------------------------------------------------------ CPU
def test_copies_equal_rejects_wrong_problems_and_one_ulp():
    """The comparison rejects a batch whose problem b was read from b +- 1, 32, 128 or 256,
    and one whose partial last copy is one ulp off in one element."""
    g = torch.Generator().manual_seed(0)
    base = torch.randn(6, K, 3, generator=g, dtype=F64)
    B = 1000
    big = tile(base, 1, B, K)
    assert first_mismatch(big, base, K, 1) is None
    for s in (1, -1, 32, -32, 128, -128, 256, -256):
        shifted = big.index_select(1, (torch.arange(B) + s) % B)
        assert first_mismatch(shifted, base, K, 1) is not None, s
    b = B - 1                            # in the partial last copy
    assert B % K != 0
    off = big.clone()
    off[4, b, 2] = torch.nextafter(off[4, b, 2], torch.tensor(float("inf"), dtype=F64))
    assert first_mismatch(off, base, K, 1) == b
    with pytest.raises(AssertionError, match="problem %d " % b):
        copies_equal(off, base, K, 1, "u")
    c = CASES["lindx4+2-T200"]           # its C really is past 2^31 elements
    assert c["T"] * c["Bs"][0] * (c["ns"] + c["nc"]) ** 2 > 2 ** 31


def _oracle_forward(port, name, P, dyn, k):
    c = CASES[name]
    T = c["T"]
    kw = dict(P["kw"])
    if P["F"] is not None:
        dyn = port.LinDx(P["F"], P["f"])
    return port.mpc_forward(P["x0"], port.QuadCost(_dense_C(P["C"], T, k), P["c"]), dyn, c["ns"],
                            c["nc"], T, lqr_iter=c["L"], final_pass=False, **kw)


def _select(name, P, j):
    def one(key, t):
        d = _per_problem(name, key, t)
        return t if d is None else t.narrow(d, j, 1).contiguous()
    q = {key: one(key, v) for key, v in P.items() if key not in ("kw", "W")}
    q["kw"] = {key: one(key, v) for key, v in P["kw"].items()}
    q["W"] = P["W"]
    return q


# Bases whose batch-global decisions move the oracle's result by less than the bound below:
# the single-input LinDx bases (their batch and per-problem results agree to ~1e-12: n = 1
# pnqp exits after a step or two) and rocket at lqr_iter = 4.  On these the tiled batches
# check the box, tensor-bound and u_zero_I paths at scale, not the decisions.
DECISIONS_PER_PROBLEM = {"lindx5+1-box", "lindx5+1-tensor", "lindx31+1-box", "rocket"}


@pytest.mark.parametrize("name", [n for n in BOXED if n not in DECISIONS_PER_PROBLEM])
def test_batch_decisions_are_exercised(port, name):
    """On every other boxed base the oracle's batch result differs from the per-problem
    result by more than 100x the suite's FP64 bound on one step (3e-9, test_oracle_matrix):
    the batch-global decisions (pnqp's exit and Armijo loop, the line search) change the
    result, so a tiled batch that did not make its base's decisions could not reproduce it.
    And the base problems' results are pairwise distinct, so a problem read from the wrong
    place shows."""
    P, dyn, _ = base_problem(port, name)
    o = _oracle_forward(port, name, P, dyn, K)
    d = 0.0
    for j in range(K):
        oj = _oracle_forward(port, name, _select(name, P, j), dyn, 1)
        d = max(d, rel(o.u[:, j:j + 1], oj.u), rel(o.x[:, j:j + 1], oj.x))
    assert d > 100 * 3e-9, (name, d)
    tau = torch.cat((o.x, o.u), 2).transpose(0, 1).reshape(K, -1)
    dist = torch.cdist(tau, tau) + torch.eye(K, dtype=F64)
    assert float(dist.min()) > 0


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
    """The family of every solve_mpc call from here on."""
    seen = []
    orig = sol.solve_mpc

    def recorded(*a, **kw):
        out = orig(*a, **kw)
        seen.append(family(out[3]))
        return out

    monkeypatch.setattr(sol, "solve_mpc", recorded)
    return seen


@pytest.fixture
def dthetas(sol, monkeypatch):
    """The per-problem dtheta [B, n_theta] of every DiLQR backward from here on (its caller
    sums it over the batch)."""
    seen = []
    orig = sol.dilqr_backward

    def recorded(*a, **kw):
        out = orig(*a, **kw)
        seen.append(out[2])
        return out

    monkeypatch.setattr(sol, "dilqr_backward", recorded)
    return seen


def fresh_stream(sol, dev):
    """A stream with no workspace yet (torch reuses stream handles: drop a cached one)."""
    s = torch.cuda.Stream(device=dev)
    sol._ws_cache.pop((dev.index if dev.index is not None else 0, s.cuda_stream), None)
    return s


def _capacity(name, dtype):
    c = CASES[name]
    lib = _lib()
    dyn = lib.DYN_ROCKET if c.get("env") == "rocket" else lib.DYN_LINDX
    return group_capacity(c["ns"], c["nc"], dyn, dtype)


# ------------------------------------------------------------------ forward solves
@pytest.mark.gpu
@pytest.mark.parametrize("name,dtype,Bspec", _fwd_params())
def test_forward_tiled(sol, dilqr, port, dev, name, dtype, Bspec):
    """x, u, costs, K, k of every copy equal the base solve's bit for bit; the pnqp counts of
    every iteration are the base's."""
    c = CASES[name]
    cap = _capacity(name, dtype) if isinstance(Bspec, str) or Bspec == 257 else None
    B = resolve_B(Bspec, cap)
    assert B % K != 0                    # the last copy is partial
    if cap is not None:                  # the regime each B is meant to run
        if Bspec == 257:
            assert -(-B // (GROUP_THREADS // GROUP_LANES)) <= cap // GROUP_THREADS
        elif Bspec in ("cap/16+1", "cap"):
            assert -(-B // (GROUP_THREADS // GROUP_LANES)) > cap // GROUP_THREADS
    need_memory(solve_bytes(B, c["T"], c["ns"], c["nc"], dtype), name)
    P, _, pdx = base_problem(port, name)
    base = solve(sol, dilqr, name, on_device(name, P, dtype, dev), dtype, dev, pdx)
    big = solve(sol, dilqr, name, on_device(name, P, dtype, dev, B), dtype, dev, pdx)
    assert family(base[3]) == family_of(name, dtype, K, cap)
    assert family(big[3]) == family_of(name, dtype, B, cap)
    assert big[3].qp_iters == base[3].qp_iters
    outs = lambda o: (("x", o[0], 1), ("u", o[1], 1), ("costs", o[2], 0), ("K", o[3].K, 1),
                      ("k", o[3].k, 1))
    if cap is not None and B > cap:
        # another family than the base's: copies bitwise among themselves, the base within
        # the bound by which the group sweep and the thread kernels agree
        tol = 1e-9 if dtype == F64 else 1e-4
        for (nm, v, dim), (_, r, _) in zip(outs(big), outs(base)):
            copies_equal(v, v.narrow(dim, 0, K), K, dim, nm)
            assert rel(v.narrow(dim, 0, K), r) < tol, (nm, rel(v.narrow(dim, 0, K), r))
        print("\n[tiled] %s B=%d replay retries %d" % (name, B, big[3].retries))
    else:
        for (nm, v, dim), (_, r, _) in zip(outs(big), outs(base)):
            copies_equal(v, r, K, dim, nm)
    if cap is not None:
        print("\n[tiled] %s %s capacity %d" % (name, dtype, cap))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_base_vs_oracle(sol, dilqr, port, dev, name):
    """Each base in FP64 end to end against port.mpc_forward: 1e-6 (test_env_vs_oracle's
    bound), the first iteration's pnqp count exact.  eps = 0 runs every base past its
    convergence, where the line search compares costs that tie to the last bit, so the later
    iterations' counts of two correct implementations may differ."""
    c = CASES[name]
    P, dyn, pdx = base_problem(port, name)
    x, u, costs, info = solve(sol, dilqr, name, on_device(name, P, F64, dev), F64, dev, pdx)
    o = _oracle_forward(port, name, P, dyn, K)
    assert o.n_iters == c["L"]
    err = max(rel(x, o.x), rel(u, o.u), rel(costs, o.costs))
    print("\n[tiled] %s base vs oracle %.2e" % (name, err))
    assert err < 1e-6
    assert info.qp_iters[0] == o.qp_iters[0]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("n", [4, 33])
def test_pnqp_tiled(dilqr, port, dev, n, dtype):
    """pnqp.pnqp, batch-global: x, the free set, the factorisation and the iteration count
    of every copy equal the base's (n = 4 compiled, n = 33 runtime kernels)."""
    pnqp = importlib.import_module("differentiable-ilqr_b200.pnqp")
    lib = _lib()
    assert pnqp.kernels(dtype, n, 20) == (lib.PNQP_COMPILED if n == 4 else lib.PNQP_RT)
    g = torch.Generator().manual_seed(n)
    A = torch.randn(K, n, n, generator=g, dtype=F64)
    H = A.transpose(1, 2) @ A + 0.5 * torch.eye(n, dtype=F64)
    q = 2 * torch.randn(K, n, generator=g, dtype=F64)
    lo = -torch.rand(K, n, generator=g, dtype=F64)
    hi = torch.rand(K, n, generator=g, dtype=F64)
    args = [t.to(dev, dtype) for t in (H, q, lo, hi)]
    x, fac, If, i = dilqr.pnqp(*args)
    X, FAC, IF, I = dilqr.pnqp(*[tile(t, 0, B_FULL, K).contiguous() for t in args])
    assert I == i
    fac = fac if isinstance(fac, tuple) else (fac,)
    FAC = FAC if isinstance(FAC, tuple) else (FAC,)
    for nm, big, base in zip(("x", "If", "lu", "piv"), (X, IF) + FAC, (x, If) + fac):
        copies_equal(big, base, K, 0, nm)
    if dtype == F64:                     # the base against the oracle (test_pnqp_standalone)
        o = port.pnqp(H, q, lo, hi)
        assert i == o.n_iter and torch.equal(If.cpu(), o.If) and rel(x, o.x) < 1e-12




# ------------------------------------------------------------------ gradients
def _upstream(shapes, seed, dtype, dev):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(sh, generator=g, dtype=F64).to(dev, dtype) for sh in shapes]


@pytest.mark.gpu
@pytest.mark.parametrize("bcast", [False, True], ids=["dense", "C_n"])
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("name", ["lindx5+1-box", "lindx8+4-box", "lindx7+3-box"])
def test_kkt_tiled(dilqr, port, dev, families, name, dtype, bcast):
    """KKT gradients through mpc.MPC at B = 65541: dx_init, dF, df (and dC, dc of a dense cost)
    of every copy equal the base's bit for bit.  With C[n,n] / c[n] the gradient is a batch sum:
    it is compared with sum_j m_j g_j, g_j the dense per-problem gradient of the base."""
    c = CASES[name]
    ns, nc, T = c["ns"], c["nc"], c["T"]
    n = ns + nc
    B = B_FULL
    need_memory(2 * solve_bytes(B, T, ns, nc, dtype), name)
    P, _, _ = base_problem(port, name)

    def run(Bn, cost):
        d = on_device(name, P, dtype, dev, None if Bn == K else Bn)
        if cost == "bcast":
            Cin, cin = d["C"][0, 0].clone(), d["c"][0, 0].clone()
        elif cost == "dense_of_bcast":
            Cin = d["C"][0, 0].expand(T, Bn, n, n).contiguous()
            cin = d["c"][0, 0].expand(T, Bn, n).contiguous()
        else:
            Cin, cin = d["C"], d["c"]
        leaves = [t.clone().requires_grad_() for t in (d["x0"], Cin, cin, d["F"], d["f"])]
        m = dilqr.MPC(ns, nc, T, lqr_iter=c["L"], eps=0.0, verbose=-1, exit_unconverged=False,
                      detach_unconverged=False, n_batch=Bn, u_lower=-BOX, u_upper=BOX)
        x, u, _ = m(leaves[0], dilqr.QuadCost(leaves[1], leaves[2]), dilqr.LinDx(leaves[3], leaves[4]))
        assert m.last_info.n_iters == c["L"]
        gx, gu = _upstream(((T, K, ns), (T, K, nc)), 12, dtype, dev)
        if Bn != K:
            gx, gu = tile(gx, 1, Bn, K), tile(gu, 1, Bn, K)
        ((x * gx).sum() + (u * gu).sum()).backward()
        return x.detach(), u.detach(), [t.grad for t in leaves], gx, gu, m.last_info.qp_iters

    cost = "bcast" if bcast else "dense"
    xb, ub, gb, gxb, gub, qb = run(K, cost)
    xB, uB, gB, _, _, qB = run(B, cost)
    assert qB == qb
    fam = [expected_family(ns, nc, dtype, True), expected_family(ns, nc, dtype, False)]
    assert families == fam * 2
    copies_equal(xB, xb, K, 1, "x")
    copies_equal(uB, ub, K, 1, "u")
    for nm, got, want, dim in zip(("dx0", "dC", "dc", "dF", "df"), gB, gb, (0, 1, 1, 1, 1)):
        if bcast and nm in ("dC", "dc"):
            continue
        copies_equal(got, want, K, dim, nm)
    if bcast:
        _, _, gd, _, _, _ = run(K, "dense_of_bcast")
        m = copy_counts(B, K)
        assert_batch_sum(gB[1], gd[1].sum(0), m, SUM_TOL[dtype], "dC")
        assert_batch_sum(gB[2], gd[2].sum(0), m, SUM_TOL[dtype], "dc")
    elif dtype == F64:                   # the base against the oracle at its own solution
        up = lambda t: t.detach().cpu().double()
        kk = port.kkt_backward(up(gxb), up(gub), P["x0"], P["C"], P["c"], P["F"], P["f"], up(xb),
                               up(ub), ns, nc, u_lower=-BOX, u_upper=BOX)
        for got, r, nm in zip(gb, (kk.dx_init, kk.dC, kk.dc, kk.dF, kk.df), ("dx0", "dC", "dc", "dF", "df")):
            assert rel(got, r) < 1e-10, (nm, rel(got, r))


def _env_bounds(name, pdx, T, k):
    """Per-problem [T,k,1] bounds (test_dilqr_backward_paths._bounds): the active sets differ."""
    g = torch.Generator().manual_seed(31)
    s = torch.tensor((1.0, 0.5, 0.15), dtype=F64)
    up = s[torch.randint(0, 3, (k,), generator=g)]
    lo = s[torch.randint(0, 3, (k,), generator=g)]
    ramp = 1.0 + 0.1 * torch.linspace(0, 1, T, dtype=F64)[:, None]
    up = torch.where(up < 1, up * ramp, up)
    lo = torch.where(lo < 1, lo * ramp, lo)
    return (pdx.lower * lo)[..., None].contiguous(), (pdx.upper * up)[..., None].contiguous()


DILQR_CASES = [("cartpole", 50, 65536, "scalar", "fused"), ("cartpole", 50, B_FULL, "scalar", "fused"),
               ("pendulum", 20, B_FULL, "tensor", "generic")]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("name,T,B,bounds,path", DILQR_CASES,
                         ids=["%s-%d-%s" % (c[0], c[2], c[4]) for c in DILQR_CASES])
def test_dilqr_tiled(dilqr, port, dev, families, dthetas, name, T, B, bounds, path, dtype):
    """The DiLQR implicit gradient through mpc_explicit.MPC with a dense cost: dC, dc and the
    per-problem dtheta [B, n_theta] of every copy equal the base's bit for bit; theta.grad is
    their batch sum.  The FP32 cartpole base (41 problems, an odd batch) is also the test of
    the final adjoint pass's bulk stores, whose destination is misaligned there."""
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    ns, nc = (5, 1) if name == "cartpole" else (3, 1)
    need_memory(3 * solve_bytes(B, T, ns, nc, dtype), name)
    pdx, x0, C, cv, kw = env_problem(port, name, T, K, F64, sigma=0.5, seed=3)
    if name == "cartpole":
        x0 = importlib.import_module("bench").make_inputs(torch, K, F64, 3)[0]
    lo, hi = (pdx.lower, pdx.upper) if bounds == "scalar" else _env_bounds(name, pdx, T, K)
    del kw["u_lower"], kw["u_upper"]
    kw["eps"] = 0.0
    cls = env.CartpoleDx if name == "cartpole" else env.PendulumDx

    def run(Bn):
        t = (lambda v, dim: v.to(dev, dtype).contiguous()) if Bn == K else \
            (lambda v, dim: tile(v.to(dev, dtype), dim, Bn, K).contiguous())
        lb, ub = (lo, hi) if bounds == "scalar" else (t(lo, 1), t(hi, 1))
        theta = pdx.params.to(dev, dtype).requires_grad_()
        Cg, cg = t(C, 1).requires_grad_(), t(cv, 1).requires_grad_()
        m = dilqr.mpc_explicit.MPC(ns, nc, T, u_lower=lb, u_upper=ub, lqr_iter=10, verbose=-1,
                                   exit_unconverged=False, detach_unconverged=False,
                                   richardson_passes=4, richardson_tol=None, n_batch=Bn, **kw)
        x, u, _ = m(t(x0, 0), dilqr.QuadCost(Cg, cg), cls(theta))
        assert m.last_info.n_iters == 10
        gx, gu = _upstream(((T, K, ns), (T, K, nc)), 11, dtype, dev)
        if Bn != K:
            gx, gu = tile(gx, 1, Bn, K), tile(gu, 1, Bn, K)
        ((x * gx).sum() + (u * gu).sum()).backward()
        st = m.last_backward
        assert (st["fused"], st["factored"]) == ((True, True) if path == "fused" else (False, False))
        return x.detach(), u.detach(), Cg.grad, cg.grad, dthetas[-1], theta.grad, m.last_info.qp_iters

    base, big = run(K), run(B)
    # the two forward solves (and, on the generic path, its line-searching adjoint solves)
    assert len(families) >= 2 and set(families) == {"thread"}
    assert big[6] == base[6]
    for nm, got, want, dim in zip(("x", "u", "dC", "dc", "dtheta"), big[:5], base[:5], (1, 1, 1, 1, 0)):
        copies_equal(got, want, K, dim, nm)
    assert base[4].shape == (K, len(pdx.params))
    assert_batch_sum(big[5], base[4], copy_counts(B, K), SUM_TOL[dtype], "theta.grad")


IL_CASES = [(1, True), (4, True), (4, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("n_rich,tiled", IL_CASES, ids=["r1-tile", "r4-tile", "r4-bcast"])
def test_imitation_step_tiled(dilqr, sol, dev, families, dthetas, n_rich, tiled, dtype):
    """The benchmarked step (il.ImitationStep, cartpole T = 50, lqr_iter = 10) at B = 65536:
    its [dtheta, dq, dp, loss] is sum_j m_j (contribution of j), the contributions from a base
    run of mpc_explicit.MPC with a dense cost and the upstream gradient 2 (u - u_exp) / (T B nc)
    of the big batch.  Three steps on one stream, which reuse the trace guess and the gains
    guess, equal each other and a step on a fresh stream bit for bit."""
    if dtype == F32 and not tiled:
        pytest.skip("the broadcast-cost step is checked in FP64")
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    il = importlib.import_module("differentiable-ilqr_b200.il")
    bench = importlib.import_module("bench")
    T, B, ns, nc = bench.T_H, 65536, bench.NS, bench.NC
    n = ns + nc
    need_memory(3 * solve_bytes(B, T, ns, nc, dtype), "imitation step")
    x0, uexp = [t.to(dev, dtype) for t in bench.make_inputs(torch, K, F64, 5)]
    proto = env.CartpoleDx()
    q, p = [t.to(dev, dtype) for t in proto.get_true_obj()]
    theta = torch.tensor(bench.THETA, dtype=dtype, device=dev)
    X0, UEXP = tile(x0, 0, B, K).contiguous(), tile(uexp, 1, B, K).contiguous()

    flats = []
    with torch.cuda.stream(fresh_stream(sol, dev)):
        step = il.ImitationStep(env.CartpoleDx, T=T, lqr_iter=bench.LQR_ITER, dtype=dtype,
                                device=dev, n_richardson=n_rich, tile=tiled)
        res = step.prepare(X0, q, p, theta)
        for _ in range(3):
            flats.append(step.run_resident(res, UEXP).clone())
            assert step.mpc.last_info.n_iters == bench.LQR_ITER
        torch.cuda.current_stream().synchronize()
    print("\n[tiled] imitation step redone %d retries %d" % (step.redone, step.retries))
    with torch.cuda.stream(fresh_stream(sol, dev)):
        step2 = il.ImitationStep(env.CartpoleDx, T=T, lqr_iter=bench.LQR_ITER, dtype=dtype,
                                 device=dev, n_richardson=n_rich, tile=tiled)
        flats.append(step2.run_resident(step2.prepare(X0, q, p, theta), UEXP).clone())
        torch.cuda.current_stream().synchronize()
    for f in flats[1:]:
        assert torch.equal(f, flats[0])

    # the base: per-problem contributions
    Cg = torch.diag(q)[None, None].repeat(T, K, 1, 1).requires_grad_()
    cg = p[None, None].repeat(T, K, 1).requires_grad_()
    th = theta.clone().requires_grad_()
    m = dilqr.mpc_explicit.MPC(ns, nc, T, u_lower=proto.lower, u_upper=proto.upper,
                               lqr_iter=bench.LQR_ITER, verbose=-1, exit_unconverged=False,
                               detach_unconverged=False, linesearch_decay=proto.linesearch_decay,
                               max_linesearch_iter=proto.max_linesearch_iter, eps=proto.mpc_eps,
                               richardson_passes=n_rich, richardson_tol=None, n_batch=K)
    _, u, _ = m(x0, dilqr.QuadCost(Cg, cg), env.CartpoleDx(th))
    assert m.last_info.n_iters == bench.LQR_ITER
    assert m.last_info.qp_iters == step.mpc.last_info.qp_iters
    assert set(families) == {"thread"}
    d = (u - uexp).detach()
    torch.autograd.backward([u], [2.0 * d / (T * B * nc)])
    contrib = torch.cat((dthetas[-1], Cg.grad.diagonal(dim1=-2, dim2=-1).sum(0), cg.grad.sum(0),
                         (d * d).sum((0, 2))[:, None] / (T * B * nc)), 1)
    assert contrib.shape == (K, len(bench.THETA) + 2 * n + 1)
    assert_batch_sum(flats[0], contrib, copy_counts(B, K), SUM_TOL[dtype], "step")
