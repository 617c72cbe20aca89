"""pnqp of any size up to 256 variables and any iteration budget up to 1024: the runtime-dimension
pnqp kernels (dilqr_pnqp_rt, csrc/pnqp_rt.cuh).

CPU tests check the ABI: which call the library picks for (n, n_iter) and the argument checks of
dilqr_pnqp_rt.  GPU tests check that the runtime kernels return bitwise what the compiled kernels
return on the sizes both serve, that sizes and budgets without compiled kernels agree with the
CPU oracle, FP32 optimality, and a batch larger than one grid row of blocks."""
import ctypes as C
import importlib

import pytest
import torch

from common import rel


def _lib():
    return importlib.import_module("differentiable-ilqr_b200._lib")


def _pnqp_mod():
    return importlib.import_module("differentiable-ilqr_b200.pnqp")


COMPILED_N = (1, 2, 3, 4, 6, 8)


# ------------------------------------------------------------------ CPU: the C ABI
def test_pnqp_kernels_choice():
    lib = _lib()
    L = lib.lib()
    for dt in (lib.F32, lib.F64):
        for n in COMPILED_N:
            assert L.dilqr_pnqp_kernels(dt, n, 20) == lib.PNQP_COMPILED
            assert L.dilqr_pnqp_kernels(dt, n, 10) == lib.PNQP_RT
        for n, it in ((5, 20), (7, 1), (16, 20), (256, 20), (4, 1024), (256, 1024), (4, 21)):
            assert L.dilqr_pnqp_kernels(dt, n, it) == lib.PNQP_RT
        assert L.dilqr_pnqp_kernels(dt, 257, 20) == -2
        assert L.dilqr_pnqp_kernels(dt, 4, 1025) == -2
        assert L.dilqr_pnqp_kernels(dt, 0, 20) == -1
        assert L.dilqr_pnqp_kernels(dt, 4, 0) == -1
        assert L.dilqr_pnqp_kernels(dt, -3, 20) == -1
    assert L.dilqr_pnqp_kernels(7, 4, 20) == -1


def test_pnqp_limits_raise_and_name_the_limit():
    lib = _lib()
    pm = _pnqp_mod()
    with pytest.raises(lib.DilqrLibraryError, match="256 variables"):
        pm.kernels(torch.float64, 257, 20)
    with pytest.raises(lib.DilqrLibraryError, match="1024 iterations"):
        pm.kernels(torch.float32, 4, 1025)
    with pytest.raises(lib.DilqrLibraryError, match="invalid argument"):
        pm.kernels(torch.float64, 4, 0)
    assert pm.kernels(torch.float64, 4, 20) == lib.PNQP_COMPILED
    assert pm.kernels(torch.float64, 5, 20) == lib.PNQP_RT


def test_pnqp_rt_argument_checks():
    """Errors come back before anything is enqueued: the pointers are host addresses, which a
    launch would fault on."""
    lib = _lib()
    L = lib.lib()
    buf = (C.c_double * 4096)()
    base = C.addressof(buf)
    p = base + (-base) % 16

    def call(dtype=lib.F64, n=5, n_iter=20, B=4, null=None, trace=p):
        ptrs = [p] * 9 + [trace]
        if null is not None:
            ptrs[null] = None
        H, q, lo, hi, x0, x, lu, piv, If, tr = ptrs
        return L.dilqr_pnqp_rt(dtype, n, n_iter, B, H, q, lo, hi, x0, x, lu, piv, If, tr, 0, p,
                               None)

    for null in (0, 1, 2, 3, 5, 6, 7, 8, 9):    # x_init (4) may be NULL
        assert call(null=null) == -1
    assert L.dilqr_pnqp_rt(lib.F64, 5, 20, 4, p, p, p, p, None, p, p, p, p, p, 0, None, None) == -1
    assert call(dtype=5) == -1
    assert call(B=0) == -1
    assert call(n=0) == -1
    assert call(n_iter=0) == -1
    assert call(n=257) == -2
    assert call(n_iter=1025) == -2
    assert call(trace=p + 2) == -3


def test_pnqp_refuses_cpu_tensors():
    lib = _lib()
    pm = _pnqp_mod()
    H = torch.eye(5, dtype=torch.float64)[None]
    with pytest.raises(lib.DilqrLibraryError, match="CUDA"):
        pm.pnqp(H, torch.zeros(1, 5, dtype=torch.float64), -1.0, 1.0)


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def box_qp(n, B, seed, warm):
    """Well-conditioned H = A'A/n + I, boxes that make constraints active."""
    g = torch.Generator().manual_seed(1000 * n + seed)
    f64 = torch.float64
    A = torch.randn(B, n, n, generator=g, dtype=f64)
    H = A.transpose(1, 2) @ A / n + torch.eye(n, dtype=f64)
    q = 2 * torch.randn(B, n, generator=g, dtype=f64)
    lo = -torch.rand(B, n, generator=g, dtype=f64)
    hi = torch.rand(B, n, generator=g, dtype=f64)
    x0 = torch.randn(B, n, generator=g, dtype=f64) if warm else None
    return H, q, lo, hi, x0


def _dev(t, dev, dtype=torch.float64):
    return None if t is None else t.to(dev, dtype)


def _check_oracle(port, H, q, lo, hi, x0, out, n_iter=20):
    """The assertions of test_gpu_parity.test_pnqp_standalone."""
    x, fac, If, i = out
    o = port.pnqp(H, q, lo, hi, x_init=x0, n_iter=n_iter)
    assert i == o.n_iter
    assert torch.equal(If.cpu(), o.If)                       # active sets: exact
    assert rel(x, o.x) < 1e-12
    B, n = q.shape
    rhs = torch.randn(B, n, 1, generator=torch.Generator().manual_seed(11), dtype=torch.float64)
    want = torch.linalg.solve(o.Hfree, rhs)
    if n == 1:
        got = rhs.to(x.device) / fac
    else:
        got = torch.linalg.lu_solve(fac[0], fac[1], rhs.to(x.device))
    assert rel(got, want) < 1e-10
    return o


@pytest.mark.gpu
@pytest.mark.parametrize("solo", [False, True], ids=["global", "solo"])
@pytest.mark.parametrize("warm", [False, True], ids=["cold", "warm"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", COMPILED_N)
def test_runtime_equals_compiled_bitwise(dev, n, dtype, warm, solo):
    """On the compiled sizes dilqr_pnqp_rt returns bitwise what dilqr_pnqp returns: same
    solution, free set, factor, pivots, iteration count and trace re-runs.  B = 70 leaves a
    partial last warp of the compiled kernel."""
    lib = _lib()
    pm = _pnqp_mod()
    H, q, lo, hi, x0 = box_qp(n, 70, seed=1, warm=warm)
    args = [_dev(t, dev, dtype) for t in (H, q, lo, hi, x0)]
    xc, fc, Ifc, ic, stc, runs_c = pm.run(*args, solo=solo, kind=lib.PNQP_COMPILED)
    xr, fr, Ifr, ir, str_, runs_r = pm.run(*args, solo=solo, kind=lib.PNQP_RT)
    assert torch.equal(xc, xr)
    assert torch.equal(Ifc, Ifr)
    if n == 1:
        assert torch.equal(fc, fr)
    else:
        assert torch.equal(fc[0], fr[0]) and torch.equal(fc[1], fr[1])
    assert ic == ir and stc.pnqp_unconverged == str_.pnqp_unconverged
    assert runs_c == runs_r
    if warm and not solo:
        assert runs_r > 1       # the batch-global replay had to correct its guess


@pytest.mark.gpu
@pytest.mark.parametrize("warm", [False, True], ids=["cold", "warm"])
@pytest.mark.parametrize("n", [5, 7, 16, 31, 32, 33, 64, 100, 256])
def test_uncompiled_sizes_against_oracle(dilqr, port, dev, n, warm):
    B = 70 if n <= 33 else (16 if n <= 100 else 6)
    H, q, lo, hi, x0 = box_qp(n, B, seed=2, warm=warm)
    out = dilqr.pnqp(*[_dev(t, dev) for t in (H, q, lo, hi, x0)])
    o = _check_oracle(port, H, q, lo, hi, x0, out)
    assert (o.If == 0).any()                                 # some bound is active


@pytest.mark.gpu
@pytest.mark.parametrize("n_iter", [1, 5, 50])
@pytest.mark.parametrize("n", [4, 7, 64])
def test_iteration_budget_against_oracle(dilqr, port, dev, n, n_iter):
    B = 70 if n <= 7 else 16
    H, q, lo, hi, x0 = box_qp(n, B, seed=3, warm=True)
    out = dilqr.pnqp(*[_dev(t, dev) for t in (H, q, lo, hi, x0)], n_iter=n_iter)
    _check_oracle(port, H, q, lo, hi, x0, out, n_iter=n_iter)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 33])
def test_exhausted_budget_warns(dilqr, port, dev, capsys, n):
    """A warm start away from the solution is still moving after one iteration: i = n_iter - 1
    and the reference's warning."""
    pm = _pnqp_mod()
    H, q, lo, hi, x0 = box_qp(n, 32, seed=4, warm=True)
    args = [_dev(t, dev) for t in (H, q, lo, hi, x0)]
    _, _, _, i, st, _ = pm.run(*args, n_iter=1)
    assert i == 0 and st.pnqp_unconverged != 0
    capsys.readouterr()
    out = dilqr.pnqp(*args, n_iter=1)
    assert out[3] == 0
    assert "[WARNING] pnqp warning: Did not converge" in capsys.readouterr().out
    _check_oracle(port, H, q, lo, hi, x0, out, n_iter=1)


@pytest.mark.gpu
@pytest.mark.parametrize("warm", [False, True], ids=["cold", "warm"])
@pytest.mark.parametrize("n", [5, 16, 64, 256])
def test_fp32_uncompiled_sizes(dilqr, port, dev, n, warm):
    """FP32: the projected gradient of the box QP vanishes to FP32 accuracy and x is close to
    the FP64 oracle."""
    B = 64 if n <= 64 else 6
    H, q, lo, hi, x0 = box_qp(n, B, seed=5, warm=warm)
    x, _, If, i = dilqr.pnqp(*[_dev(t, dev, torch.float32) for t in (H, q, lo, hi, x0)])
    assert x.dtype == torch.float32 and If.dtype == torch.float32
    xd = x.cpu().double()
    g = (H @ xd.unsqueeze(2)).squeeze(2) + q
    resid = (xd - torch.minimum(torch.maximum(xd - g, lo), hi)).abs().max()
    assert float(resid) < 1e-4 * (1 + float(q.abs().max()))
    o = port.pnqp(H, q, lo, hi, x_init=x0)
    assert rel(x, o.x) < 1e-4


@pytest.mark.gpu
def test_solo_large_batch(dev):
    """solo: every problem on its own, so the first 64 problems of B = 65541 equal a 64-problem
    call bitwise (the grid has more than one row of blocks and a partial last block)."""
    pm = _pnqp_mod()
    B = 65541
    H, q, lo, hi, x0 = box_qp(7, B, seed=6, warm=True)
    args = [_dev(t, dev) for t in (H, q, lo, hi, x0)]
    x, (lu, piv), If, _, _, _ = pm.run(*args, solo=True)
    xs, (lus, pivs), Ifs, _, _, _ = pm.run(*[a[:64].contiguous() for a in args], solo=True)
    assert torch.equal(x[:64], xs) and torch.equal(If[:64], Ifs)
    assert torch.equal(lu[:64], lus) and torch.equal(piv[:64], pivs)
    assert torch.isfinite(x).all()
    assert bool(((x >= args[2]) & (x <= args[3])).all())
