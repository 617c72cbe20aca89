"""``pnqp`` -- drop-in for the reference's projected-Newton box QP (pnqp.py:5-82):
``pnqp(H, q, lower, upper, x_init=None, n_iter=20) -> (x, H_or_LU, If, i)`` with the
reference's batch-global termination / Armijo semantics (see DESIGN.md section 3).
Any size n <= 256 and budget n_iter <= 1024: the library serves n in {1,2,3,4,6,8} with
n_iter = 20 from compiled kernels, everything else from the runtime-dimension kernels."""
import ctypes as C

import torch

from . import _lib
from ._solver import _DT, _ptr, _stream


def pnqp(H, q, lower, upper, x_init=None, n_iter=20, solo=False):
    x, fac, If, i, st, _ = run(H, q, lower, upper, x_init, n_iter, solo)
    if st.pnqp_unconverged:
        print("[WARNING] pnqp warning: Did not converge")          # pnqp.py:81
    return x, fac, If, i


def kernels(dtype, n, n_iter):
    """Which call serves pnqp of size n with budget n_iter (the library's choice):
    ``_lib.PNQP_COMPILED`` (dilqr_pnqp) or ``_lib.PNQP_RT`` (dilqr_pnqp_rt)."""
    kind = _lib.lib().dilqr_pnqp_kernels(_DT[dtype], n, n_iter)
    if kind == -2:
        raise _lib.DilqrLibraryError(
            "pnqp n=%d n_iter=%d is not supported: the pnqp kernels take at most %d variables "
            "and %d iterations" % (n, n_iter, _lib.PNQP_RT_MAX_N, _lib.PNQP_RT_MAX_ITER))
    if kind < 0:
        _lib.check(kind, "dilqr_pnqp_kernels(n=%d, n_iter=%d)" % (n, n_iter))
    return kind


def run(H, q, lower, upper, x_init=None, n_iter=20, solo=False, kind=None):
    """pnqp without the warning: returns ``(x, fac, If, i, status, runs)``, ``runs`` the
    number of kernel runs the trace replay took.  ``kind`` forces a family
    (``_lib.PNQP_RT`` serves every size); None takes the library's choice."""
    if not H.is_cuda:
        raise _lib.DilqrLibraryError("pnqp runs on CUDA tensors only")
    B, n, _ = H.shape
    dtype, dev = H.dtype, H.device
    if kind is None:
        kind = kernels(dtype, n, n_iter)
    Hc = H.detach().contiguous()
    qc = q.detach().contiguous()

    def bound(v):
        if isinstance(v, float):
            return torch.full((B, n), v, dtype=dtype, device=dev)
        return v.detach().to(dtype).expand(B, n).contiguous()

    lo, hi = bound(lower), bound(upper)
    x0 = None if x_init is None else x_init.detach().contiguous()
    x = torch.empty(B, n, dtype=dtype, device=dev)
    lu = torch.empty(B, n, n, dtype=dtype, device=dev)
    piv = torch.empty(B, n, dtype=torch.int32, device=dev)
    If = torch.empty(B, n, dtype=dtype, device=dev)
    trace = torch.zeros(2 * n_iter, dtype=torch.int32, device=dev)
    status_dev = torch.zeros(64, dtype=torch.uint8, device=dev)
    args = (_ptr(Hc), _ptr(qc), _ptr(lo), _ptr(hi), _ptr(x0), _ptr(x), _ptr(lu), _ptr(piv),
            _ptr(If), _ptr(trace), 1 if solo else 0, _ptr(status_dev), _stream())
    # A run replays word `it` exactly at most three runs after the words before it (a wrong
    # guess goes 0 -> "moving, first Armijo pass exits" -> "moving, no pass exits" -> the
    # observed word), and one more run confirms the whole trace, so the runs grow with n_iter:
    # 3 n_iter + 2 suffice; 3 n_iter + 4 is the bound of 64 runs at the default budget.
    for runs in range(1, 3 * n_iter + 5):
        if kind == _lib.PNQP_COMPILED:
            _lib.call("dilqr_pnqp", _DT[dtype], n, B, *args)
        else:
            _lib.call("dilqr_pnqp_rt", _DT[dtype], n, n_iter, B, *args)
        st = _lib.DilqrStatus.from_buffer_copy(status_dev.cpu().numpy().tobytes())
        if st.trace_match or solo:
            break
    else:
        raise _lib.DilqrLibraryError("pnqp control-flow trace did not stabilise")
    i = int(st.n_total_qp_iter) - 1
    fac = lu if n == 1 else (lu, piv)
    return x, fac, If, i, st, runs
