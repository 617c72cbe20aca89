"""Host driver of the fused iLQR kernels: owns the workspace, drives the
iLQR outer loop of ``MPC.forward`` (reference mpc.py:184-337) over the C ABI,
and assembles the KKT gradients (reference lqr_step.py:312-407).

Nothing here computes on the CPU; torch is used for device memory, streams and
autograd plumbing only.
"""
import ctypes as C

import torch

from . import _lib

_DT = {torch.float32: _lib.F32, torch.float64: _lib.F64}


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _on_device_of(argname, pos):
    """Run the wrapped entry point with the device of its tensor argument current, so
    the stream the kernels are enqueued on (``_stream``), the workspace and the operands
    always belong to the same GPU, whatever the caller's current device is."""
    import functools

    def deco(fn):
        @functools.wraps(fn)
        def wrapped(*args, **kw):
            t = kw.get(argname) if argname in kw else (args[pos] if len(args) > pos else None)
            if torch.is_tensor(t) and t.is_cuda:
                with torch.cuda.device(t.device):
                    return fn(*args, **kw)
            return fn(*args, **kw)
        return wrapped
    return deco


class DynSpec:
    """What the rollouts integrate: LinDx tensors or an env_dx model id + theta."""

    def __init__(self, kind, params=None, F=None, f=None, aux=None, ai=None):
        self.kind = kind
        self.params = list(params) if params is not None else []
        self.F = F
        self.f = f
        self.aux = aux      # DYN_NN / DYN_NN_RT: packed weight buffer (device tensor)
        self.ai = list(ai) if ai is not None else []


class SolveInfo:
    def __init__(self):
        self.n_iters = 0
        self.retries = 0
        self.qp_iters = []
        self.log = []
        self.pnqp_unconverged = 0
        self.converged = False
        self.full_du_norm = None


MAX_PIPELINED_ITERS = 1024


class Deferred:
    """Validation reads of a step, postponed to ONE host synchronisation at its end.

    The solver's control flow never needs the host in the common case (the stop rule, the
    pnqp trace check and the adjoint line-search test all run on the device); the host only
    has to learn *afterwards* that nothing went wrong.  Each `add` enqueues a small D2H
    copy into pinned memory behind the kernels that produce the data; `resolve` waits once
    and runs the checks.  A failed check means the optimistic launches behind it computed
    on a stale guess: the caller repeats the step with immediate checks."""

    _pool = {}

    def __init__(self):
        self.items = []
        self.ok = True
        self.reasons = []

    def add(self, dev_bytes, fn):
        n = dev_bytes.numel()
        key = (n, len(self.items))
        host = Deferred._pool.get(key)
        if host is None:
            host = torch.empty(n, dtype=torch.uint8).pin_memory()
            Deferred._pool[key] = host
        host.copy_(dev_bytes, non_blocking=True)
        self.items.append((host, fn))

    def resolve(self):
        if self.items:
            torch.cuda.current_stream().synchronize()
        for host, fn in self.items:
            why = fn(host.numpy().tobytes())
            if why:
                self.ok = False
                self.reasons.append(why)
        self.items = []
        return self.ok


class Workspace:
    """Device scratch + status / control blocks for one (shape, dtype) family; reused."""

    def __init__(self, nbytes, device):
        self.gen = 0       # bumped by every solve that (re)uses the buffer
        self.gains_guess = None   # (shape key) the gains sweep's own trace guess is valid for
        self.solve_guess = None   # (shape key) of the solve whose final trace guess is in place
        self.buf = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=device)
        self.status_dev = torch.zeros(64, dtype=torch.uint8, device=device)
        self.status_host = torch.zeros(64, dtype=torch.uint8).pin_memory()
        # pipelined outer loop: [control block | one status block per iteration]
        self.pipe_dev = torch.zeros(64 * (1 + MAX_PIPELINED_ITERS), dtype=torch.uint8, device=device)
        self.pipe_host = torch.zeros(64 * (1 + MAX_PIPELINED_ITERS), dtype=torch.uint8).pin_memory()


_ws_cache = {}


def _require_cuda(t, name):
    if not t.is_cuda:
        raise _lib.DilqrLibraryError(
            "%s must be a CUDA tensor: this package has no CPU path" % name)


def _aligned(t):
    """TMA slabs start on 16-byte boundaries: re-materialise views that do not."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _contig(t):
    return t if t is None or t.is_contiguous() else t.contiguous()


def cost_layout(t, T, B, tail_ndim):
    """Classify a cost tensor handed to the solver (mpc.py:205-219 accepts C[n,n],
    C[T,n,n], C[T,B,n,n] and expands with stride 0).  Returns (mode, base) with
    mode 0: dense [T,B,..] contiguous; 1: batch-broadcast, base [T,..]; 2: base [..]."""
    t = t.detach()
    if t.ndimension() == tail_ndim:
        return 2, t.contiguous()
    if t.ndimension() == tail_ndim + 1:
        return 1, t.contiguous()
    st = t.stride()
    if t.shape[1] > 1 and st[1] == 0:
        if st[0] == 0:
            return 2, t[0, 0].contiguous()
        return 1, t[:, 0].contiguous()
    return 0, t.contiguous()


def dense_cost(t, T, B, tail_ndim):
    """Materialise any accepted cost layout as [T,B,..] (generic / LinDx-KKT paths)."""
    t = t.detach()
    if t.ndimension() == tail_ndim:
        t = t.unsqueeze(0).unsqueeze(0)
    elif t.ndimension() == tail_ndim + 1:
        t = t.unsqueeze(1)
    return t.expand(T, B, *t.shape[2:]).contiguous()


def lindx_kernels(dtype, n_state, n_ctrl):
    """The dynamics id whose kernels serve a LinDx problem of this shape (the library's
    choice: the compiled kernels where they exist, else the runtime-dimension ones)."""
    kind = _lib.lib().dilqr_lindx_kernels(_DT[dtype], n_state, n_ctrl)
    if kind == -2:
        raise _lib.DilqrLibraryError(
            "LinDx n_state=%d n_ctrl=%d is not supported: the LinDx kernels take at most 32 "
            "variables (n_state + n_ctrl)" % (n_state, n_ctrl))
    if kind < 0:
        _lib.check(kind, "dilqr_lindx_kernels")
    return kind


def nn_kernels(dtype, n_state, n_ctrl):
    """The dynamics id whose kernels serve a network (NNDynamics) problem of this shape: the
    compiled kernels where they exist, else the runtime-dimension ones."""
    kind = _lib.lib().dilqr_nn_kernels(_DT[dtype], n_state, n_ctrl)
    if kind == -2:
        raise _lib.DilqrLibraryError(
            "NNDynamics n_state=%d n_ctrl=%d is not supported: the network kernels take at most "
            "32 variables (n_state + n_ctrl)" % (n_state, n_ctrl))
    if kind < 0:
        _lib.check(kind, "dilqr_nn_kernels")
    return kind


def _make_problem(x_init, C_, c_, dyn, n_state, n_ctrl, T, u_lower, u_upper, u_zero_I,
                  linesearch_decay, max_linesearch_iter, best_cost_eps, gain_solve,
                  solo, delta_u=None):
    L = _lib.lib()
    _require_cuda(x_init, "x_init")
    dtype = x_init.dtype
    if dtype not in _DT:
        raise _lib.DilqrLibraryError("dtype %s unsupported (float32/float64 only)" % dtype)
    B = x_init.shape[0]
    s = _lib.DilqrSolve()
    s.n_state, s.n_ctrl, s.T, s.n_batch = n_state, n_ctrl, T, B
    s.dtype = _DT[dtype]
    if dyn.kind == _lib.DYN_LINDX:
        s.dynamics = lindx_kernels(dtype, n_state, n_ctrl)
    elif dyn.kind == _lib.DYN_NN:
        s.dynamics = nn_kernels(dtype, n_state, n_ctrl)
    else:   # an explicit id, e.g. a runtime family forced on a compiled shape
        s.dynamics = dyn.kind
    s.gain_solve = gain_solve
    s.solo = int(solo)   # 0 batch-global, 1 per-problem QP flags, 2 per-problem outer loop too
    s.max_linesearch_iter = max_linesearch_iter
    s.linesearch_decay = float(linesearch_decay)
    s.best_cost_eps = float(best_cost_eps)
    for i, v in enumerate(dyn.params):
        s.dyn_params[i] = float(v)
    keep = []  # keep tensors alive while kernels run

    def dev(t, name, dt=dtype):
        if t is None:
            return None
        _require_cuda(t, name)
        t = _contig(t.detach().to(dt))
        keep.append(t)
        return t

    xi = dev(x_init, "x_init")
    _require_cuda(C_, "C")
    _require_cuda(c_, "c")
    s.C_bcast, Cd = cost_layout(C_.to(dtype), T, B, 2)
    s.c_bcast, cd = cost_layout(c_.to(dtype), T, B, 1)
    keep.extend((Cd, cd))
    s.x_init, s.C, s.c = _ptr(xi), _ptr(Cd), _ptr(cd)
    if dyn.kind in (_lib.DYN_NN, _lib.DYN_NN_RT):
        aux = dev(dyn.aux, "network weights")
        s.dyn_aux = _ptr(aux)
        for i, v in enumerate(dyn.ai):
            s.dyn_ai[i] = int(v)
    if dyn.kind in (_lib.DYN_LINDX, _lib.DYN_LINDX_RT):
        Fd = dev(dyn.F, "F")
        fd = dev(dyn.f, "f") if (dyn.f is not None and dyn.f.nelement() > 0) else None
        s.F, s.f = _ptr(Fd), _ptr(fd)
        s.has_f = 1 if fd is not None else 0
    if u_lower is None:
        s.bounds_kind = _lib.BOUNDS_NONE
    elif isinstance(u_lower, float) and isinstance(u_upper, float):
        s.bounds_kind = _lib.BOUNDS_SCALAR
        s.u_lower, s.u_upper = u_lower, u_upper
    else:
        s.bounds_kind = _lib.BOUNDS_TENSOR
        lo = u_lower if torch.is_tensor(u_lower) else torch.full(
            (T, B, n_ctrl), float(u_lower), dtype=dtype, device=x_init.device)
        hi = u_upper if torch.is_tensor(u_upper) else torch.full(
            (T, B, n_ctrl), float(u_upper), dtype=dtype, device=x_init.device)
        lo = dev(lo.expand(T, B, n_ctrl), "u_lower")
        hi = dev(hi.expand(T, B, n_ctrl), "u_upper")
        s.u_lower_t, s.u_upper_t = _ptr(lo), _ptr(hi)
    if delta_u is not None:
        assert u_lower is not None               # lqr_step.py:195
        s.delta_u, s.has_delta_u = float(delta_u), 1
    if u_zero_I is not None:
        zi = dev(u_zero_I.expand(T, B, n_ctrl), "u_zero_I", torch.uint8)
        s.u_zero_I = _ptr(zi)
    # the library chooses how the iterations resolve pnqp's batch-global decisions
    rc = L.dilqr_mpc_plan(C.byref(s))
    if rc == -2:
        raise _lib.DilqrLibraryError(
            "no kernel compiled for dtype=%s n_state=%d n_ctrl=%d dynamics=%d "
            "(add it to DILQR_CONFIGS in csrc/api.cu)" % (dtype, n_state, n_ctrl, dyn.kind))
    _lib.check(rc, "dilqr_mpc_plan")
    need = L.dilqr_workspace_bytes(C.byref(s))
    # one workspace per (device, stream): solves on different streams never share scratch;
    # it only ever grows (the layout comes from the problem struct, not the buffer size)
    key = (x_init.device.index, torch.cuda.current_stream(x_init.device).cuda_stream)
    ws = _ws_cache.get(key)
    if ws is None or ws.buf.numel() < need:
        ws = None
        _ws_cache.pop(key, None)      # release the smaller buffer before allocating
        ws = Workspace(need, x_init.device)
        _ws_cache[key] = ws
    ws.gen += 1
    s.workspace = _ptr(ws.buf)
    s.workspace_bytes = ws.buf.numel()
    s.status = _ptr(ws.status_dev)
    return L, s, ws, keep


def _read_status(ws):
    ws.status_host.copy_(ws.status_dev, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return _lib.DilqrStatus.from_buffer_copy(ws.status_host.numpy().tobytes())


MAX_TRACE_RETRIES = 64


def _iterate_committed(L, s, ws, info, sync=True):
    """One iLQR iteration including the trace-verification retry loop.  With
    ``sync=False`` (no box constraints => no pnqp trace, and nothing on the host
    depends on the status) the call is fire-and-forget: no host sync."""
    st = _stream()
    for _ in range(MAX_TRACE_RETRIES):
        _lib.call("dilqr_mpc_iterate", C.byref(s), st)
        _lib.call("dilqr_mpc_commit", C.byref(s), st)
        if not sync:
            return None
        status = _read_status(ws)
        if status.trace_match:
            return status
        info.retries += 1
    raise _lib.DilqrLibraryError("pnqp control-flow trace did not stabilise")


def _fill_info(info, raw, verbose):
    """Decode [control | status x iterations] as read back from the device."""
    c = _lib.DilqrControl.from_buffer_copy(raw[:64])
    n_done = c.iters_done
    for j in range(n_done):
        stt = _lib.DilqrStatus.from_buffer_copy(raw[64 * (1 + j):64 * (2 + j)])
        info.qp_iters.append(stt.n_total_qp_iter)
        info.pnqp_unconverged += stt.pnqp_unconverged
        info.log.append((stt.n_total_qp_iter, stt.max_full_du, stt.mean_alpha, stt.mean_best_cost))
        if stt.pnqp_unconverged and verbose >= 0:
            for _ in range(stt.pnqp_unconverged):
                print("[WARNING] pnqp warning: Did not converge")   # pnqp.py:81
        info.max_full_du, info.mean_alpha = stt.max_full_du, stt.mean_alpha
        info.mean_best_cost = stt.mean_best_cost
    info.n_iters = n_done
    return c


def _solve_pipelined(L, s, ws, info, n_loops, eps_cmp, not_improved_lim, verbose, deferred=None):
    """Outer iLQR loop with the stop rule and the trace check on the device
    (DilqrControl): all iterations are enqueued back to back, ONE host sync at the
    end; a wrong pnqp trace guess halts the queue and the loop resumes from there.
    With ``deferred`` not even that: the control block is copied back asynchronously and
    checked when the caller resolves the step (a halted queue then invalidates it)."""
    st = _stream()
    ctrl = _lib.DilqrControl()
    ctrl.eps = eps_cmp
    ctrl.not_improved_lim = not_improved_lim
    ws.pipe_host[:64].copy_(torch.frombuffer(bytearray(bytes(ctrl)), dtype=torch.uint8))
    ws.pipe_dev[:64].copy_(ws.pipe_host[:64], non_blocking=True)
    base = ws.pipe_dev.data_ptr()
    s.control = C.c_void_p(base)
    start = 0
    nbytes = 64 * (1 + n_loops)
    if deferred is not None:
        for j in range(n_loops):
            s.iteration = j
            s.status = C.c_void_p(base + 64 * (1 + j))
            _lib.call("dilqr_mpc_iterate", C.byref(s), st)
            _lib.call("dilqr_mpc_commit", C.byref(s), st)

        def check(raw, info=info, verbose=verbose):
            c = _fill_info(info, raw, verbose)
            return "pnqp trace mismatch in the forward solve" if c.halt == 2 else None

        deferred.add(ws.pipe_dev[:nbytes], check)
        # finish reads the number of committed iterations from the control block
        s.iteration = n_loops - 1
        s.status = _ptr(ws.status_dev)
        return
    for _ in range(MAX_TRACE_RETRIES * 4):
        for j in range(start, n_loops):
            s.iteration = j
            s.status = C.c_void_p(base + 64 * (1 + j))
            _lib.call("dilqr_mpc_iterate", C.byref(s), st)
            _lib.call("dilqr_mpc_commit", C.byref(s), st)
        ws.pipe_host[:nbytes].copy_(ws.pipe_dev[:nbytes], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        raw = ws.pipe_host[:nbytes].numpy().tobytes()
        c = _lib.DilqrControl.from_buffer_copy(raw[:64])
        if c.halt == 2:                      # trace mismatch: redo iteration c.iters_done
            info.retries += 1
            start = c.iters_done
            ws.pipe_dev[:4].zero_()
            continue
        break
    else:
        raise _lib.DilqrLibraryError("pnqp control-flow trace did not stabilise")
    c = _fill_info(info, raw, verbose)
    s.iteration = c.iters_done - 1
    s.control = None
    s.status = _ptr(ws.status_dev)


@_on_device_of("x_init", 0)
def solve_mpc(x_init, C_, c_, dyn, n_state, n_ctrl, T, u_lower=None, u_upper=None,
              u_zero_I=None, u_init=None, lqr_iter=10, eps=1e-7, linesearch_decay=0.2,
              max_linesearch_iter=10, not_improved_lim=5, best_cost_eps=1e-4,
              gain_solve=_lib.GAIN_PLAIN, solo=False, verbose=0, x_cur=None,
              want_gains=False, sync=True, gains_only=False, pipelined=True, delta_u=None,
              deferred=None, reuse_trace=True):
    """MPC.forward (mpc.py:184-306): returns (x, u, costs, info).  With ``x_cur``
    given this is a single LQRStep around (x_cur, u_init) (lqr_step.py:277-309)
    and returns the *new* iterate."""
    L, s, ws, keep = _make_problem(x_init, C_, c_, dyn, n_state, n_ctrl, T, u_lower,
                                   u_upper, u_zero_I, linesearch_decay,
                                   max_linesearch_iter, best_cost_eps, gain_solve, solo, delta_u)
    dtype, dev = x_init.dtype, x_init.device
    B = x_init.shape[0]
    if u_init is not None:
        u0 = u_init.detach()
        if u0.ndimension() == 2:
            u0 = u0.unsqueeze(1).expand(T, B, -1)
        u0 = u0.to(dtype).contiguous()
        keep.append(u0)
        s.u_init = _ptr(u0)
    if x_cur is not None:
        xc = x_cur.detach().to(dtype).contiguous()
        keep.append(xc)
        s.x_cur = _ptr(xc)
    st = _stream()
    info = SolveInfo()
    if gains_only:
        s.gains_only = 1
        want_gains = True
    # warm-started repeats of the same solve (training loops, closed loops): the trace the
    # previous solve ended with predicts this one's first iteration better than the default
    shape_key = (s.n_state, s.n_ctrl, s.T, s.n_batch, s.dtype, s.dynamics, s.bounds_kind, int(solo))
    s.keep_trace_guess = 1 if (reuse_trace and u_init is not None and x_cur is None
                               and ws.solve_guess == shape_key) else 0
    ws.solve_guess = shape_key if x_cur is None else None
    _lib.call("dilqr_mpc_begin", C.byref(s), st)
    # python float eps is compared in the data dtype by torch (mpc.py:299)
    eps_cmp = float(torch.tensor(eps, dtype=dtype))
    n_not_improved = 0
    n_loops = 1 if x_cur is not None else lqr_iter
    nosync = (not sync) and n_loops == 1 and (s.bounds_kind == _lib.BOUNDS_NONE or solo)
    if int(solo) == 2 and n_loops > 1 and not n_loops <= MAX_PIPELINED_ITERS:
        raise ValueError("solo=2 needs lqr_iter <= %d" % MAX_PIPELINED_ITERS)
    if n_loops > 1 and n_loops <= MAX_PIPELINED_ITERS and (
            (pipelined and verbose <= 0) or int(solo) == 2):
        if int(solo) == 2:
            deferred = None          # its host logic needs the statuses right away
        _solve_pipelined(L, s, ws, info, n_loops, eps_cmp, not_improved_lim, verbose, deferred)
        n_loops = 0
    for i in range(n_loops):
        s.iteration = i
        status = _iterate_committed(L, s, ws, info, sync=not nosync)
        info.n_iters = i + 1
        if status is None:
            break
        info.qp_iters.append(status.n_total_qp_iter)
        info.pnqp_unconverged += status.pnqp_unconverged
        info.log.append((status.n_total_qp_iter, status.max_full_du, status.mean_alpha,
                         status.mean_best_cost))
        if status.pnqp_unconverged and verbose >= 0:
            for _ in range(status.pnqp_unconverged):
                print("[WARNING] pnqp warning: Did not converge")   # pnqp.py:81
        n_not_improved += 1                                          # mpc.py:266
        if i > 0 and status.any_improved:
            n_not_improved = 0                                       # mpc.py:281
        if verbose > 0:
            print("| %d | %.4e | %.2e | %.2e | %d |" % (
                i, status.mean_best_cost, status.max_full_du, status.mean_alpha,
                status.n_total_qp_iter))
        info.max_full_du = status.max_full_du
        info.mean_alpha = status.mean_alpha
        info.mean_best_cost = status.mean_best_cost
        if status.max_full_du < eps_cmp or n_not_improved > not_improved_lim:
            break                                                    # mpc.py:299-301
    x = u = costs = du = None
    if not gains_only:
        x = torch.empty(T, B, n_state, dtype=dtype, device=dev)
        u = torch.empty(T, B, n_ctrl, dtype=dtype, device=dev)
        costs = torch.empty(B, dtype=dtype, device=dev)
        du = torch.empty(B, dtype=dtype, device=dev)
        s.x_out, s.u_out, s.cost_out, s.du_out = _ptr(x), _ptr(u), _ptr(costs), _ptr(du)
    extra = {}
    if x_cur is not None and not gains_only:
        al = torch.empty(B, dtype=dtype, device=dev)
        s.alpha_out = _ptr(al)
        extra["alphas"] = al
    if want_gains:
        K = torch.empty(T, B, n_ctrl, n_state, dtype=dtype, device=dev)
        k = torch.empty(T, B, n_ctrl, dtype=dtype, device=dev)
        s.K_out, s.k_out = _ptr(K), _ptr(k)
        extra["K"], extra["k"] = K, k
    _lib.call("dilqr_mpc_finish", C.byref(s), st)
    s.control = None
    # what the backward pass can pick up from this solve while the workspace is untouched
    info._problem = (s, ws, ws.gen, keep + [t for t in (x, u) if t is not None])
    info.full_du_norm = du
    info.converged = None
    for k_, v_ in extra.items():
        setattr(info, k_, v_)
    return x, u, costs, info


@_on_device_of("x", 3)
def kkt_grads(C_, c_, F, x, u, dx, du, r, n_state, n_ctrl, want_df=True, want_dF=True):
    """Costate recursions + outer products (lqr_step.py:343-404)."""
    L = _lib.lib()
    T, B = x.shape[0], x.shape[1]
    dtype, dev = x.dtype, x.device
    k = _lib.DilqrKkt()
    k.n_state, k.n_ctrl, k.T, k.n_batch, k.dtype = n_state, n_ctrl, T, B, _DT[dtype]
    k.dynamics = lindx_kernels(dtype, n_state, n_ctrl)
    ten = [_contig(t.detach()) for t in (C_, c_, F, x, u, dx, du, r)]
    k.C, k.c, k.F, k.x, k.u, k.dx, k.du, k.r = [_ptr(t) for t in ten]
    n = n_state + n_ctrl
    dC = torch.empty(T, B, n, n, dtype=dtype, device=dev)
    dc = torch.empty(T, B, n, dtype=dtype, device=dev)
    dF = torch.empty(max(T - 1, 0), B, n_state, n, dtype=dtype, device=dev) if want_dF else None
    df = torch.empty(max(T - 1, 0), B, n_state, dtype=dtype, device=dev) if want_df else None
    dx0 = torch.empty(B, n_state, dtype=dtype, device=dev)
    k.dC, k.dc, k.dF, k.df, k.dx_init = _ptr(dC), _ptr(dc), _ptr(dF), _ptr(df), _ptr(dx0)
    _lib.call("dilqr_kkt_grads", C.byref(k), _stream())
    return dx0, dC, dc, dF, df


@_on_device_of("x_init", 2)
def kkt_backward(dl_dx, dl_du, x_init, C_, c_, F, f, x, u, n_state, n_ctrl, u_lower=None,
                 u_upper=None, gain_solve=_lib.GAIN_PLAIN, back_eps=1e-7):
    """LQRStepFn.backward (lqr_step.py:312-407): adjoint LQR solve with the
    active controls pinned to zero, then the gradient assembly."""
    T, B = x.shape[0], x.shape[1]
    r = torch.cat((dl_dx, dl_du), 2).contiguous()
    if u_lower is None:
        I = None
    else:                                                   # lqr_step.py:325-326
        I = (torch.abs(u - u_lower) <= 1e-8) | (torch.abs(u - u_upper) <= 1e-8)
    zero = torch.zeros_like(x_init)
    dyn = DynSpec(_lib.DYN_LINDX, F=F, f=None)
    dx, du, _, _ = solve_mpc(zero, C_, -r, dyn, n_state, n_ctrl, T, u_zero_I=I, lqr_iter=1,
                             eps=back_eps, gain_solve=gain_solve, verbose=-1, sync=False)
    want_df = f is not None and f.nelement() > 0
    return kkt_grads(C_, c_, F, x, u, dx, du, r, n_state, n_ctrl, want_df)


def _adjoint_struct(kind, n_state, n_ctrl, T, B, dtype, u_lower, u_upper, theta, Cb, cb):
    a = _lib.DilqrAdjoint()
    a.n_state, a.n_ctrl, a.T, a.n_batch, a.dtype, a.dynamics = n_state, n_ctrl, T, B, _DT[dtype], kind
    a.bounds_kind = _lib.BOUNDS_NONE if u_lower is None else _lib.BOUNDS_SCALAR
    a.gain_solve = _lib.GAIN_CHOL_REG
    a.C_bcast, a.c_bcast = Cb, cb
    if u_lower is not None:
        a.u_lower, a.u_upper = u_lower, u_upper
    for i in range(8):
        a.dyn_params[i] = theta[i]
    return a


FUSED_BACKWARD = True      # A/B knob: False restores the round-1 kernel sequence


@_on_device_of("x_init", 0)
def dilqr_prepare(x_init, C_, c_, x, u, dxmod, n_state, n_ctrl, u_lower=None, u_upper=None,
                  solo=False, theta_host=None, factored=True, solve_info=None, deferred=None):
    """Everything of the DiLQR backward that depends only on the forward solution
    (x*, u*), the cost and theta -- NOT on the upstream gradient: the gains of the final
    no-op LQR pass (lqr_step_explicit.py:604-618), the primal costates with the
    contracted second-order tables, and the factorisation of the adjoint LQR solves.
    ``MPC.forward`` enqueues this right behind the solve when a gradient will be asked
    for, so the device works through it while the host is busy with the loss and the
    autograd dispatch.

    ``solve_info``: the SolveInfo of the forward solve.  While its workspace is untouched
    the fused sequence is used (pendulum / cartpole, scalar bounds): ONE sweep over the
    solver's own outputs gives gains + costates (``dilqr_mpc_gains``, C from the packed
    workspace copy), the second-order tables are a (t, problem)-parallel kernel
    (``dilqr_lam_tables``), and the factorisation reads the packed C as well -- no
    re-layout of the trajectory, no gather of the gains, C streamed 2 x 21 instead of
    3 x 36 scalars per (t, problem)."""
    T, B = x.shape[0], x.shape[1]
    dtype, dev = x.dtype, x.device
    n = n_state + n_ctrl
    kind = dxmod._dilqr_kind
    # theta_host: the host copy the forward pass already fetched (saves a device sync)
    theta = dxmod._theta() if theta_host is None else (C.c_double * 8)(
        *(list(theta_host) + [0.0] * (8 - len(theta_host))))
    x = x.detach().contiguous()
    u = u.detach().contiguous()
    scalar_bounds = u_lower is None or (isinstance(u_lower, float) and isinstance(u_upper, float))
    if not scalar_bounds or kind == _lib.DYN_ROCKET:
        factored = False      # factored adjoint kernels: pendulum / cartpole only
    # cost layout: dense [T,B,..] or broadcast (C[n,n] / C[T,n,n]); the generic path
    # (LinDx kernels + kkt_grads) wants dense tensors.  C_sum / c_sum: the axes the
    # densification of a C[n,n] / C[T,n,n] added, over which the backward sums the dense
    # gradient so that it comes back in the shape handed in (as the factored path's does)
    C_in, c_in = C_, c_
    Cb, C_ = cost_layout(C_in.to(dtype), T, B, 2)
    cb, c_ = cost_layout(c_in.to(dtype), T, B, 1)
    C_sum = c_sum = ()
    if not factored and (Cb or cb):
        C_, c_ = dense_cost(C_in.to(dtype), T, B, 2), dense_cost(c_in.to(dtype), T, B, 1)
        C_sum = {2: (0, 1), 3: (1,)}.get(C_in.dim(), ())
        c_sum = {1: (0, 1), 2: (1,)}.get(c_in.dim(), ())
        Cb = cb = 0
    prep = dict(theta=theta, kind=kind, factored=factored, Cb=Cb, cb=cb, C_=C_, c_=c_, x=x, u=u,
                x_init=x_init, C_in=C_in, c_in=c_in, C_sum=C_sum, c_sum=c_sum, fused=False)
    nW = (B + 31) // 32
    fused = (FUSED_BACKWARD and factored and solve_info is not None and n_ctrl == 1
             and getattr(solve_info, "_problem", None) is not None)
    if fused:
        sp, ws, gen, keep = solve_info._problem
        fused = ws.gen == gen and sp.x_out is not None and sp.u_zero_I is None
    if fused:
        L = _lib.lib()
        view = _lib.DilqrWsView()
        _lib.check(L.dilqr_workspace_view(C.byref(sp), C.byref(view)), "dilqr_workspace_view")
        lam = torch.empty(T, nW, n_state, 32, dtype=dtype, device=dev)
        sp.status = _ptr(ws.status_dev)
        sp.control = None

        def gains_ok(raw):
            st = _lib.DilqrStatus.from_buffer_copy(raw)
            return None if st.trace_match else "pnqp trace mismatch in the final LQR pass"

        shape_key = (sp.n_state, sp.n_ctrl, sp.T, sp.n_batch, sp.dtype, sp.dynamics)
        for attempt in range(MAX_TRACE_RETRIES):
            sp.gains_guess_reset = 0 if ws.gains_guess == shape_key else 1
            ws.gains_guess = shape_key
            rc = _lib.call("dilqr_mpc_gains", C.byref(sp), _ptr(lam), _stream(), allow=(-2,))
            if rc == -2:
                fused = False      # shape without the fused sweep: round-1 sequence below
                break
            if deferred is not None:
                deferred.add(ws.status_dev, gains_ok)
                break
            # the trace guess was the last iteration's; a wrong guess has been corrected on
            # the device: run the sweep again
            if gains_ok(bytes(_read_status_raw(ws))) is None:
                break
            if solve_info is not None:
                solve_info.retries += 1
        else:
            raise _lib.DilqrLibraryError("pnqp control-flow trace did not stabilise")
    if fused:
        nlam = _lib.lib().dilqr_lam_pack_size(kind)
        Lam = torch.empty(T - 1, nW, nlam, 32, dtype=dtype, device=dev)
        _lib.call("dilqr_lam_tables", _DT[dtype], kind, theta, T, B, _ptr(x), _ptr(u), _ptr(lam),
                  _ptr(Lam), _stream())
        a = _adjoint_struct(kind, n_state, n_ctrl, T, B, dtype, u_lower, u_upper, theta, Cb, cb)
        resid = torch.zeros(3, dtype=torch.float64, device=dev)
        a.C, a.x, a.u, a.Lam = _ptr(C_), _ptr(x), _ptr(u), _ptr(Lam)
        a.Cpk, a.cpk_state = view.Cpk, view.cpk_state
        a.resid = _ptr(resid)
        need = L.dilqr_adjoint_workspace_bytes(C.byref(a))
        aws = torch.empty(need, dtype=torch.uint8, device=dev)
        a.workspace, a.workspace_bytes = _ptr(aws), need
        _lib.call("dilqr_adjoint_factor", C.byref(a), _stream())
        prep.update(fused=True, a=a, ws=aws, resid=resid, lam=lam, Lam=Lam, Kk=view.Kk,
                    solver_ws=ws, solver_gen=gen, keep=keep,
                    dtau_off=L.dilqr_adjoint_dtau_offset(C.byref(a)))
        return prep
    # ---- round-1 sequence (any env_dx model, tensor bounds, foreign workspaces) ----------
    # (1) gains of the final no-op LQR pass at tau* (lqr_step_explicit.py:604-618)
    dyn = DynSpec(kind, params=list(theta))
    _, _, _, info = solve_mpc(x_init, C_in, c_in, dyn, n_state, n_ctrl, T, u_lower=u_lower,
                              u_upper=u_upper, u_init=u, x_cur=x, lqr_iter=1, max_linesearch_iter=1,
                              solo=solo, verbose=-1, gains_only=True)
    K = info.K
    # (2) primal costates + contracted second-order tables
    lam = torch.empty(T, B, n_state, dtype=dtype, device=dev)
    if factored:   # packed, warp-blocked Lam (only the structurally non-zero entries)
        nlam = _lib.lib().dilqr_lam_pack_size(kind)
        Lam = torch.empty(T - 1, nW, nlam, 32, dtype=dtype, device=dev)
    else:
        Lam = torch.empty(T - 1, B, n, n, dtype=dtype, device=dev)
    _lib.call("dilqr_costate_tables", _DT[dtype], kind, theta, T, B, _ptr(C_), _ptr(c_), _ptr(x),
              _ptr(u), _ptr(lam), _ptr(Lam), Cb, cb, 1 if factored else 0, _stream())
    prep.update(K=K, lam=lam, Lam=Lam)
    if factored:
        # (3a) factor the adjoint LQR solves once (csrc/adjoint_kernels.cuh)
        a = _adjoint_struct(kind, n_state, n_ctrl, T, B, dtype, u_lower, u_upper, theta, Cb, cb)
        resid = torch.zeros(3, dtype=torch.float64, device=dev)
        a.C, a.x, a.u, a.Lam = _ptr(C_), _ptr(x), _ptr(u), _ptr(Lam)
        a.resid = _ptr(resid)
        need = _lib.lib().dilqr_adjoint_workspace_bytes(C.byref(a))
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        a.workspace, a.workspace_bytes = _ptr(ws), need
        _lib.call("dilqr_adjoint_factor", C.byref(a), _stream())
        prep.update(a=a, ws=ws, resid=resid)
    return prep


def _read_status_raw(ws):
    ws.status_host.copy_(ws.status_dev, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return ws.status_host.numpy().tobytes()


RICHARDSON_WARN = 1e-6     # relative residual above which a fixed-pass solve warns

# GMRES for the adjoint system (solver="gmres"): relative residual |g - A'w| / |g| per problem at
# which a problem is frozen, by dtype, and the default budget of Arnoldi steps per problem,
# GMRES_ITER_PER_DIM * T * n: full GMRES reaches the exact solution within T * n steps in exact
# arithmetic, and the factor leaves room for restarted cycles (restart < T * n) and rounding.
GMRES_TOL = {torch.float64: 1e-12, torch.float32: 1e-5}
GMRES_ITER_PER_DIM = 2


class GmresResult:
    """Per-problem outcome of ``_gmres``: iterations (int32 [B]) and final relative residual
    (float64 [B]) on the host once resolved, the operator applications enqueued, and the
    solution w [T,B,n] (device)."""

    def __init__(self, tol, max_iter, restart):
        self.tol, self.max_iter, self.restart = tol, max_iter, restart
        self.iters = self.resid = self.w = None
        self.op_calls = 0

    @property
    def unconverged(self):
        return int((~(self.resid <= self.tol)).sum())

    @property
    def worst(self):
        return float(self.resid.max()) if self.resid.numel() else 0.0

    def fill(self, raw, B):
        self.resid = torch.frombuffer(bytearray(raw[:8 * B]), dtype=torch.float64)
        self.iters = torch.frombuffer(bytearray(raw[8 * B:12 * B]), dtype=torch.int32)

    def warn(self):
        bad = self.unconverged
        if bad:
            import warnings
            warnings.warn("DiLQR backward: GMRES left %d of %d problems above the relative residual "
                          "%.1e within %d iterations (worst %.2e); their gradient is approximate -- "
                          "raise gmres_max_iter or gmres_restart"
                          % (bad, self.resid.numel(), self.tol, self.max_iter, self.worst))


def _gmres(op, op_in, op_out, negate, gx, gu, T, B, n_state, n_ctrl, restart, tol, max_iter,
           deferred=None):
    """Restarted GMRES(restart) for A'w = g per problem (include/dilqr.h, DilqrKrylov): returns
    (w[T,B,n], GmresResult).  ``op()`` applies M': reads op_in, writes op_out.  Immediate mode
    reads the count of problems still iterating once per cycle and stops when it is 0;
    ``deferred`` enqueues the whole budget with no host read (frozen problems do not change,
    so both give the same bits) and reads the per-problem status when the caller resolves it."""
    L = _lib.lib()
    dtype, dev = gu.dtype, gu.device
    n = n_state + n_ctrl
    k = _lib.DilqrKrylov()
    k.n_state, k.n_ctrl, k.T, k.n_batch, k.dtype = n_state, n_ctrl, T, B, _DT[dtype]
    k.restart = max(1, min(int(restart), T * n))
    k.max_iter = int(max_iter)
    k.op_negate = 1 if negate else 0
    k.tol = float(tol)
    w = torch.empty(T, B, n, dtype=dtype, device=dev)
    status = torch.empty(12 * B, dtype=torch.uint8, device=dev)   # resid f64 [B] | iters i32 [B]
    ctl = torch.zeros(2, dtype=torch.int32, device=dev)
    k.gx, k.gu, k.w = _ptr(gx), _ptr(gu), _ptr(w)
    k.op_in, k.op_out = _ptr(op_in), _ptr(op_out)
    k.resid = C.c_void_p(status.data_ptr())
    k.iters = C.c_void_p(status.data_ptr() + 8 * B)
    k.control = _ptr(ctl)
    need = L.dilqr_krylov_workspace_bytes(C.byref(k))
    if need == 0:
        raise _lib.DilqrLibraryError("GMRES: invalid sizes (restart %d, max_iter %d)"
                                     % (k.restart, k.max_iter))
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    k.workspace, k.workspace_bytes = _ptr(ws), need
    res = GmresResult(k.tol, k.max_iter, k.restart)
    res.w = w
    st = _stream()

    def apply():
        op()
        res.op_calls += 1

    _lib.call("dilqr_krylov_start", C.byref(k), st)
    cycle = 0
    steps = L.dilqr_krylov_cycle_steps(C.byref(k), 0)
    if steps > 0:
        apply()
    while steps > 0:
        if deferred is None and int(ctl[0]) == 0:     # every problem frozen
            break
        for j in range(steps):
            k.step = j
            _lib.call("dilqr_krylov_arnoldi", C.byref(k), st)
            if j < steps - 1:
                apply()
        _lib.call("dilqr_krylov_update", C.byref(k), st)
        apply()
        _lib.call("dilqr_krylov_restart", C.byref(k), st)
        cycle += 1
        steps = L.dilqr_krylov_cycle_steps(C.byref(k), cycle)
        if steps > 0:
            apply()
    if deferred is not None:
        def check(raw, res=res, B=B):
            res.fill(raw, B)
            res.warn()
            return None
        deferred.add(status, check)
    else:
        res.fill(status.cpu().numpy().tobytes(), B)
        res.warn()
    return w, res


@_on_device_of("x_init", 2)
def dilqr_backward(dl_dx, dl_du, x_init, C_, c_, x, u, dxmod, n_state, n_ctrl, u_lower=None,
                   u_upper=None, n_passes=8, tol=None, back_eps=1e-7, solo=False, stats=None,
                   theta_host=None, factored=True, prep=None, tile_reduce=False, deferred=None,
                   solver="richardson", gmres_restart=64, gmres_tol=None, gmres_max_iter=None):
    """DiLQR implicit gradient (lqr_step_explicit.py:652-712 + fix_point_equ
    458-598) in matrix-free form (SURVEY Appendix C; derivation in
    csrc/dilqr_backward.cuh).  Returns (dC, dc, dtheta[B, n_theta]); with
    ``tile_reduce`` the first two are instead (dq[n], dp[n]), the gradient of the tiled
    diagonal cost C[t,b] = diag(q), c[t,b] = p of il_env.py:159-162, accumulated inside the
    final adjoint pass (the dense dC / dc are never written).

    ``dl_dx`` may be None (loss independent of x): the kernels read the two halves of the
    upstream gradient separately, nothing is concatenated or copied.

    n_passes Richardson passes solve A' w = g (each = one adjoint LQR solve); with
    ``tol`` the loop stops early once max|dw| <= tol * max|w| (one host sync per
    pass).  The adjoint solves follow mpc_backup / lqr_step_backup (Cholesky +
    1e-6 I for unconstrained multi-input problems, lqr_step_backup.py:202-205).

    ``factored=True`` runs the adjoint solves with the factor-once / affine-pass
    kernels (csrc/adjoint_kernels.cuh); if any problem's adjoint step would have been
    rejected by the reference's line search (non-convex model), the whole backward is
    recomputed with the generic line-searching kernels (``factored=False``).

    ``prep``: the gradient-independent part (``dilqr_prepare``) if the forward pass
    already enqueued it.

    ``solver="gmres"`` solves A'w = g by restarted GMRES(``gmres_restart``, clipped to T n)
    per problem instead (``_gmres``), to the relative residual ``gmres_tol`` (None:
    ``GMRES_TOL`` of the dtype) within ``gmres_max_iter`` Arnoldi steps (None:
    ``GMRES_ITER_PER_DIM`` T n); ``n_passes`` / ``tol`` are then unused.  It returns the
    reference's dense solution where Richardson iteration diverges (rho(M) >= 1), at a
    data-dependent number of adjoint solves and (restart + 1) T B n scalars of basis.  A
    problem that misses the tolerance raises a warning.  When the reference's line search
    would shorten an adjoint step the adjoint map is not linear and no Krylov method applies:
    that raises ``DilqrLibraryError``."""
    if solver not in ("richardson", "gmres"):
        raise ValueError("solver must be 'richardson' or 'gmres', got %r" % (solver,))
    gmres = solver == "gmres"
    gm_opts = dict(solver=solver, gmres_restart=gmres_restart, gmres_tol=gmres_tol,
                   gmres_max_iter=gmres_max_iter)
    if prep is None:
        prep = dilqr_prepare(x_init, C_, c_, x, u, dxmod, n_state, n_ctrl, u_lower, u_upper,
                             solo, theta_host, factored)
    T, B = x.shape[0], x.shape[1]
    dtype, dev = x.dtype, x.device
    n = n_state + n_ctrl
    kind, theta, factored = prep["kind"], prep["theta"], prep["factored"]
    Cb, cb, C_d, c_d = prep["Cb"], prep["cb"], prep["C_"], prep["c_"]
    x, u, lam, Lam = prep["x"], prep["u"], prep["lam"], prep["Lam"]
    fused = prep.get("fused", False)
    if fused and prep["solver_ws"].gen != prep["solver_gen"]:
        # another solve has reused the solver workspace since: the gains / packed C the
        # fused kernels would read are gone -- recompute the preparation
        prep = dilqr_prepare(x_init, C_, c_, x, u, dxmod, n_state, n_ctrl, u_lower, u_upper,
                             solo, theta_host, factored)
        return dilqr_backward(dl_dx, dl_du, x_init, C_, c_, x, u, dxmod, n_state, n_ctrl,
                              u_lower, u_upper, n_passes, tol, back_eps, solo, stats, theta_host,
                              factored, prep, tile_reduce, deferred, **gm_opts)
    if dl_du is None:
        dl_du = torch.zeros(T, B, n_ctrl, dtype=dtype, device=dev)
    gu = _aligned(dl_du.contiguous())
    gx = None if dl_dx is None else _aligned(dl_dx.contiguous())
    passes = 0
    rel = None
    nth = len(dxmod.params)
    nwarp = (B + 31) // 32
    reduce_in_kernel = tile_reduce and factored and not Cb and not cb
    if reduce_in_kernel:
        dC = dc = None
        red = torch.empty(nwarp, 2 * n, dtype=dtype, device=dev)
    else:
        # gradients of a broadcast cost come back as per-warp partial sums (summed below)
        dC = torch.empty({0: (T, B, n, n), 1: (T, nwarp, n, n), 2: (nwarp, n, n)}[Cb], dtype=dtype,
                         device=dev)
        dc = torch.empty({0: (T, B, n), 1: (T, nwarp, n), 2: (nwarp, n)}[cb], dtype=dtype, device=dev)
    resid = prep["resid"] if factored else torch.zeros(3, dtype=torch.float64, device=dev)

    def converged():
        r = resid.cpu()
        return float(r[0]) / (float(r[1]) + 1e-300)

    krylov = None
    if gmres:
        gm_tol = GMRES_TOL[dtype] if gmres_tol is None else float(gmres_tol)
        gm_iter = GMRES_ITER_PER_DIM * T * n if gmres_max_iter is None else int(gmres_max_iter)
    if factored and gmres:
        a = prep["a"]
        st = _stream()
        # M'v: one adjoint pass with g = 0, in place on the operator buffer
        opbuf = torch.empty(T, B, n, dtype=dtype, device=dev)
        zu = torch.zeros(T, B, n_ctrl, dtype=dtype, device=dev)

        def op():
            a.gx, a.gu, a.w = None, _ptr(zu), _ptr(opbuf)
            a.first_pass, a.want_resid = 0, 0
            _lib.call("dilqr_adjoint_pass", C.byref(a), st)

        w, krylov = _gmres(op, opbuf, opbuf, False, gx, gu, T, B, n_state, n_ctrl, gmres_restart,
                           gm_tol, gm_iter, deferred)
        a.gx, a.gu, a.w = _ptr(gx), _ptr(gu), _ptr(w)
        a.first_pass = 0
    elif factored:
        a = prep["a"]
        w = torch.empty(T, B, n, dtype=dtype, device=dev) if n_passes > 0 else None
        a.gx, a.gu, a.w = _ptr(gx), _ptr(gu), _ptr(w)
        a.want_resid = 1 if tol is not None else 0
        st = _stream()
        for i in range(n_passes):
            a.first_pass = 1 if i == 0 else 0
            # the last pass of a fixed-count solve also measures how far w still moves
            if tol is None and i == n_passes - 1:
                a.want_resid = 1
            _lib.call("dilqr_adjoint_pass", C.byref(a), st)
            passes += 1
            if tol is not None:
                rel = converged()
                if rel <= tol:
                    break
        a.first_pass = 1 if passes == 0 else 0
    if factored:
        if fused:
            df = torch.empty(T - 1, nwarp, n_state, 32, dtype=dtype, device=dev)
            a.df_blk, a.df, a.dx_out, a.du_out = _ptr(df), None, None, None
        else:
            df = torch.empty(T - 1, B, n_state, dtype=dtype, device=dev)
            dxa = torch.empty(T, B, n_state, dtype=dtype, device=dev)
            dua = torch.empty(T, B, n_ctrl, dtype=dtype, device=dev)
            a.df_blk, a.df, a.dx_out, a.du_out = None, _ptr(df), _ptr(dxa), _ptr(dua)
        if reduce_in_kernel:
            a.reduce_tile, a.red_out, a.dC, a.dc = 1, _ptr(red), None, None
        else:
            a.reduce_tile, a.red_out, a.dC, a.dc = 0, None, _ptr(dC), _ptr(dc)
        _lib.call("dilqr_adjoint_final", C.byref(a), st)
    else:
        # generic path: every adjoint solve is a full (line-searching) LQR step
        g = torch.cat((gx if gx is not None else torch.zeros(T, B, n_state, dtype=dtype, device=dev),
                       gu), 2).contiguous()
        w = g.clone()
        df = torch.empty(T - 1, B, n_state, dtype=dtype, device=dev)
        F = torch.empty(T - 1, B, n_state, n, dtype=dtype, device=dev)
        _lib.call("dilqr_linearize", _DT[dtype], kind, theta, T, B, _ptr(x), _ptr(u), _ptr(F), None,
                  _stream())
        if u_lower is None:
            I = None
        else:                                               # lqr_step_explicit.py:690-691
            I = (torch.abs(u - u_lower) <= 1e-8) | (torch.abs(u - u_upper) <= 1e-8)
        negw = -g
        zero = torch.zeros_like(x_init)
        lin = DynSpec(_lib.DYN_LINDX, F=F, f=None)

        def adjoint():
            return solve_mpc(zero, C_d, negw, lin, n_state, n_ctrl, T, u_zero_I=I, lqr_iter=1,
                             eps=back_eps, gain_solve=_lib.GAIN_CHOL_REG, verbose=-1,
                             sync=False)[:2]

        if gmres:
            # M'v: the adjoint solve on cost (C, -v), then w <- 0 - Lam dtau
            vneg = torch.empty(T, B, n, dtype=dtype, device=dev)
            mv = torch.empty(T, B, n, dtype=dtype, device=dev)
            g0 = torch.zeros(T, B, n, dtype=dtype, device=dev)
            scratch = torch.empty(T, B, n, dtype=dtype, device=dev)
            res0 = torch.zeros(3, dtype=torch.float64, device=dev)

            def op():
                dxo, duo = solve_mpc(zero, C_d, vneg, lin, n_state, n_ctrl, T, u_zero_I=I,
                                     lqr_iter=1, eps=back_eps, gain_solve=_lib.GAIN_CHOL_REG,
                                     verbose=-1, sync=False)[:2]
                _lib.call("dilqr_richardson_update", _DT[dtype], n_state, n_ctrl, T, B, _ptr(g0),
                          _ptr(Lam), _ptr(dxo), _ptr(duo), _ptr(mv), _ptr(scratch), _ptr(res0),
                          _stream())

            w, krylov = _gmres(op, vneg, mv, True, gx, gu, T, B, n_state, n_ctrl, gmres_restart,
                               gm_tol, gm_iter, deferred)
            negw = -w
        for _ in range(0 if gmres else n_passes):
            dxa, dua = adjoint()
            _lib.call("dilqr_richardson_update", _DT[dtype], n_state, n_ctrl, T, B, _ptr(g),
                      _ptr(Lam), _ptr(dxa), _ptr(dua), _ptr(w), _ptr(negw), _ptr(resid), _stream())
            passes += 1
            if tol is not None:
                rel = converged()
                if rel <= tol:
                    break
        dxa, dua = adjoint()
        _, dC, dc, _, df = kkt_grads(C_d, c_d, F, x, u, dxa, dua, w, n_state, n_ctrl, want_df=True,
                                     want_dF=False)
    # (3) dtheta through the closed-loop sensitivity rollout
    dtheta = torch.empty(B, nth, dtype=dtype, device=dev)
    if fused:
        dtau = prep["ws"][prep["dtau_off"]:]
        # adjoint form: reverse sweep, second-order tables via the packed Lam
        _lib.call("dilqr_sens_theta_adjoint", _DT[dtype], kind, theta, T, B, _ptr(x), _ptr(u),
                  C.c_void_p(prep["Kk"]), _ptr(lam), _ptr(dtau), _ptr(df), _ptr(Lam),
                  _ptr(dtheta), _stream())
    else:
        _lib.call("dilqr_sens_theta", _DT[dtype], kind, theta, T, B, _ptr(x), _ptr(u),
                  _ptr(prep["K"]), _ptr(lam), _ptr(dxa), _ptr(dua), _ptr(df), _ptr(dtheta), _stream())
    if factored:
        def check(raw, passes=passes, tol=tol, stats=stats):
            import struct
            dmax, wmax, n_rej = struct.unpack("ddq", raw)
            r = dmax / (wmax + 1e-300)
            if stats is not None and passes and stats.get("resid") is None:
                stats["resid"] = r
            if n_rej and gmres:
                return ("the reference's line search would shorten an adjoint step (a non-convex "
                        "adjoint QP): the adjoint map is not linear, so GMRES cannot solve the "
                        "system the reference assembles -- use solver='richardson'")
            if n_rej:
                return "the reference's line search would reject an adjoint step"
            if passes and tol is None and r > RICHARDSON_WARN:
                import warnings
                warnings.warn("DiLQR backward: after %d Richardson passes the adjoint iterate still "
                              "moves by %.1e (relative); the gradient is approximate -- raise "
                              "richardson_passes or set richardson_tol" % (passes, r))
            return None
        if deferred is not None:
            deferred.add(resid.view(torch.uint8), check)
        else:
            # one sync at the end: did the reference's line search reject any adjoint step?
            why = check(bytes(resid.view(torch.uint8).cpu().numpy().tobytes()))
            if why and gmres:
                raise _lib.DilqrLibraryError("DiLQR backward: " + why)
            if why:
                return dilqr_backward(dl_dx, dl_du, x_init, prep["C_in"], prep["c_in"], x, u, dxmod,
                                      n_state, n_ctrl, u_lower, u_upper, n_passes, tol, back_eps,
                                      solo, stats, theta_host=theta_host, factored=False,
                                      tile_reduce=tile_reduce)
    if stats is not None:
        stats["passes"] = passes
        stats.setdefault("resid", rel)
        if rel is not None:
            stats["resid"] = rel
        stats["factored"] = factored
        stats["fused"] = fused
        stats["solver"] = solver
        if krylov is not None:
            # the per-problem status: filled now (immediate) or when the step is resolved
            stats["gmres"] = krylov
            stats["passes"] = krylov.op_calls
    if reduce_in_kernel:
        r = red.sum(0)
        return r[:n], r[n:], dtheta
    if Cb:
        dC = dC.sum(1 if Cb == 1 else 0)
    if cb:
        dc = dc.sum(1 if cb == 1 else 0)
    if prep["C_sum"]:    # generic path on a densified C[n,n] / C[T,n,n]
        dC = dC.sum(prep["C_sum"])
    if prep["c_sum"]:
        dc = dc.sum(prep["c_sum"])
    if tile_reduce:      # the tiling's adjoint on the dense gradients (generic path)
        return (dC.diagonal(dim1=-2, dim2=-1).reshape(-1, n).sum(0),
                dc.reshape(-1, n).sum(0), dtheta)
    return dC, dc, dtheta
