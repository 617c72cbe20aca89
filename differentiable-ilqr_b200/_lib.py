"""ctypes binding of libdilqr.so (the C ABI in include/dilqr.h).

There is no CPU fallback: every op of this package goes through this library;
if it is missing the import of the op fails loudly (``DilqrLibraryError``).
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# DILQR_LIB: load another build of the same library (A/B variants, tools/build_variant.sh)
LIB_PATH = os.environ.get("DILQR_LIB") or os.path.join(_HERE, "libdilqr.so")
CSRC = os.path.join(_HERE, "csrc")

F32, F64 = 0, 1
DYN_LINDX, DYN_PENDULUM, DYN_CARTPOLE, DYN_ROCKET, DYN_NN = 0, 1, 2, 3, 4
DYN_LINDX_RT = 5        # LinDx through the runtime-dimension kernels (n_state + n_ctrl <= 32)
DYN_NN_RT = 6           # NNDynamics through the runtime-dimension kernels (n_state + n_ctrl <= 32)
GAIN_PLAIN, GAIN_CHOL_REG = 0, 1
BOUNDS_NONE, BOUNDS_SCALAR, BOUNDS_TENSOR = 0, 1, 2
PNQP_MAX_ITER = 20
PNQP_COMPILED, PNQP_RT = 0, 1   # dilqr_pnqp_kernels: dilqr_pnqp / dilqr_pnqp_rt serves the call
PNQP_RT_MAX_N, PNQP_RT_MAX_ITER = 256, 1024

ERRORS = {0: "ok", -1: "invalid argument", -2: "unsupported (dtype, n_state, n_ctrl, dynamics)",
          -3: "pointer not 16-byte aligned", -4: "workspace too small",
          -5: "CUDA launch failure", -6: "group sweep launch: batch does not fit the device"}


class DilqrLibraryError(RuntimeError):
    pass


class DilqrStatus(C.Structure):
    _fields_ = [
        ("trace_match", C.c_uint32),
        ("any_improved", C.c_uint32),
        ("n_total_qp_iter", C.c_uint32),
        ("pnqp_unconverged", C.c_uint32),
        ("max_full_du", C.c_double),
        ("mean_alpha", C.c_double),
        ("mean_best_cost", C.c_double),
        ("first_mismatch", C.c_uint32),
        ("n_active", C.c_uint32),
        ("reserved", C.c_uint32 * 4),
    ]


class DilqrControl(C.Structure):
    _fields_ = [
        ("halt", C.c_uint32), ("iters_done", C.c_uint32), ("n_not_improved", C.c_uint32),
        ("not_improved_lim", C.c_uint32), ("eps", C.c_double), ("reserved", C.c_uint32 * 10),
    ]


class DilqrSolve(C.Structure):
    _fields_ = [
        ("n_state", C.c_int32), ("n_ctrl", C.c_int32), ("T", C.c_int32),
        ("n_batch", C.c_int32),
        ("dtype", C.c_int32), ("dynamics", C.c_int32), ("gain_solve", C.c_int32),
        ("bounds_kind", C.c_int32), ("solo", C.c_int32),
        ("max_linesearch_iter", C.c_int32), ("iteration", C.c_int32),
        ("has_f", C.c_int32), ("gains_only", C.c_int32), ("C_bcast", C.c_int32),
        ("c_bcast", C.c_int32),
        ("linesearch_decay", C.c_double),
        ("u_lower", C.c_double), ("u_upper", C.c_double),
        ("best_cost_eps", C.c_double),
        ("dyn_params", C.c_double * 8),
        ("x_init", C.c_void_p), ("C", C.c_void_p), ("c", C.c_void_p),
        ("F", C.c_void_p), ("f", C.c_void_p), ("u_init", C.c_void_p),
        ("x_cur", C.c_void_p), ("u_lower_t", C.c_void_p), ("u_upper_t", C.c_void_p),
        ("u_zero_I", C.c_void_p),
        ("x_out", C.c_void_p), ("u_out", C.c_void_p), ("cost_out", C.c_void_p),
        ("du_out", C.c_void_p), ("alpha_out", C.c_void_p), ("K_out", C.c_void_p),
        ("k_out", C.c_void_p),
        ("status", C.c_void_p), ("control", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("dyn_aux", C.c_void_p), ("dyn_ai", C.c_int32 * 4),
        ("delta_u", C.c_double), ("has_delta_u", C.c_int32), ("gains_guess_reset", C.c_int32),
        ("keep_trace_guess", C.c_int32), ("group_sweep", C.c_int32),
    ]


class DilqrKkt(C.Structure):
    _fields_ = [
        ("n_state", C.c_int32), ("n_ctrl", C.c_int32), ("T", C.c_int32),
        ("n_batch", C.c_int32), ("dtype", C.c_int32), ("dynamics", C.c_int32),
        ("C", C.c_void_p), ("c", C.c_void_p), ("F", C.c_void_p),
        ("x", C.c_void_p), ("u", C.c_void_p), ("dx", C.c_void_p), ("du", C.c_void_p),
        ("r", C.c_void_p),
        ("dC", C.c_void_p), ("dc", C.c_void_p), ("dF", C.c_void_p), ("df", C.c_void_p),
        ("dx_init", C.c_void_p),
    ]


class DilqrAdjoint(C.Structure):
    _fields_ = [
        ("n_state", C.c_int32), ("n_ctrl", C.c_int32), ("T", C.c_int32), ("n_batch", C.c_int32),
        ("dtype", C.c_int32), ("dynamics", C.c_int32), ("bounds_kind", C.c_int32),
        ("gain_solve", C.c_int32), ("C_bcast", C.c_int32), ("c_bcast", C.c_int32),
        ("u_lower", C.c_double), ("u_upper", C.c_double), ("dyn_params", C.c_double * 8),
        ("C", C.c_void_p), ("x", C.c_void_p), ("u", C.c_void_p), ("gx", C.c_void_p),
        ("gu", C.c_void_p),
        ("Lam", C.c_void_p), ("w", C.c_void_p), ("dC", C.c_void_p), ("dc", C.c_void_p),
        ("df", C.c_void_p), ("dx_out", C.c_void_p), ("du_out", C.c_void_p),
        ("resid", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("Cpk", C.c_void_p), ("cpk_state", C.c_void_p), ("first_pass", C.c_int32),
        ("want_resid", C.c_int32), ("reduce_tile", C.c_int32), ("reserved0", C.c_int32),
        ("red_out", C.c_void_p), ("df_blk", C.c_void_p),
    ]


class DilqrWsView(C.Structure):
    _fields_ = [
        ("Kk", C.c_void_p), ("Cpk", C.c_void_p), ("cpk_state", C.c_void_p),
        ("n_warps", C.c_int32), ("reserved", C.c_int32),
    ]


# every symbol include/dilqr.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "dilqr_version": (C.c_char_p, []),
    "dilqr_supported": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "dilqr_lindx_kernels": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "dilqr_nn_kernels": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "dilqr_mpc_plan": (C.c_int, [C.POINTER(DilqrSolve)]),
    "dilqr_workspace_bytes": (C.c_size_t, [C.POINTER(DilqrSolve)]),
    "dilqr_mpc_begin": (C.c_int, [C.POINTER(DilqrSolve), C.c_void_p]),
    "dilqr_mpc_iterate": (C.c_int, [C.POINTER(DilqrSolve), C.c_void_p]),
    "dilqr_mpc_commit": (C.c_int, [C.POINTER(DilqrSolve), C.c_void_p]),
    "dilqr_mpc_finish": (C.c_int, [C.POINTER(DilqrSolve), C.c_void_p]),
    "dilqr_mpc_gains": (C.c_int, [C.POINTER(DilqrSolve), C.c_void_p, C.c_void_p]),
    "dilqr_workspace_view": (C.c_int, [C.POINTER(DilqrSolve), C.POINTER(DilqrWsView)]),
    "dilqr_lam_tables": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int]
                         + [C.c_void_p] * 5),
    "dilqr_sens_theta_adjoint": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int,
                                           C.c_int] + [C.c_void_p] * 9),
    "dilqr_last_iterate_launches": (C.c_int, []),
    "dilqr_adjoint_dtau_offset": (C.c_size_t, [C.POINTER(DilqrAdjoint)]),
    "dilqr_kkt_grads": (C.c_int, [C.POINTER(DilqrKkt), C.c_void_p]),
    "dilqr_linearize": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dilqr_rollout": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dilqr_env_tables": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_void_p,
                                   C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p]),
    "dilqr_pnqp": (C.c_int, [C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 10 + [C.c_int]
                   + [C.c_void_p] * 2),
    "dilqr_pnqp_kernels": (C.c_int, [C.c_int] * 3),
    "dilqr_pnqp_rt": (C.c_int, [C.c_int] * 4 + [C.c_void_p] * 10 + [C.c_int] + [C.c_void_p] * 2),
    "dilqr_costate_tables": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int]
                             + [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dilqr_lam_pack_size": (C.c_int, [C.c_int]),
    "dilqr_richardson_update": (C.c_int, [C.c_int] * 5 + [C.c_void_p] * 8),
    "dilqr_sens_theta": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int]
                         + [C.c_void_p] * 9),
    "dilqr_adjoint_workspace_bytes": (C.c_size_t, [C.POINTER(DilqrAdjoint)]),
    "dilqr_adjoint_factor": (C.c_int, [C.POINTER(DilqrAdjoint), C.c_void_p]),
    "dilqr_adjoint_pass": (C.c_int, [C.POINTER(DilqrAdjoint), C.c_void_p]),
    "dilqr_adjoint_final": (C.c_int, [C.POINTER(DilqrAdjoint), C.c_void_p]),
    "dilqr_tile_cost": (C.c_int, [C.c_int] * 4 + [C.c_void_p] * 5),
    "dilqr_tile_cost_grad_workspace_bytes": (C.c_size_t, [C.c_int]),
    "dilqr_tile_cost_grad": (C.c_int, [C.c_int] * 4 + [C.c_void_p] * 5 + [C.c_size_t, C.c_void_p]),
}

_lib = None


def build(verbose=False, extra=""):
    """Compile libdilqr.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j", str(min(9, os.cpu_count() or 1))]
    if extra:
        cmd.append("EXTRA=" + extra)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or r.returncode:
        print(r.stdout)
    if r.returncode:
        raise DilqrLibraryError("building libdilqr.so failed")
    return LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise DilqrLibraryError(
            "libdilqr.so not found at %s -- run `python -c 'import __graft_entry__ as g; "
            "g.build()'` (there is no CPU fallback)" % LIB_PATH)
    try:
        L = C.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise DilqrLibraryError("cannot load %s: %s" % (LIB_PATH, e))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(code, what):
    if code != 0:
        raise DilqrLibraryError("%s failed: %s (%d)" % (what, ERRORS.get(code, "?"), code))


# kernels enqueued per C-ABI call (memsets not counted)
KERNELS_PER_CALL = {
    "dilqr_mpc_begin": 1, "dilqr_mpc_iterate": 1, "dilqr_mpc_commit": 1,
    "dilqr_mpc_finish": 1, "dilqr_mpc_gains": 3, "dilqr_lam_tables": 1,
    "dilqr_sens_theta_adjoint": 1, "dilqr_kkt_grads": 1, "dilqr_linearize": 1, "dilqr_rollout": 1,
    "dilqr_costate_tables": 1, "dilqr_richardson_update": 1, "dilqr_sens_theta": 1,
    "dilqr_adjoint_factor": 1, "dilqr_adjoint_pass": 1, "dilqr_adjoint_final": 1,
    "dilqr_pnqp": 2, "dilqr_pnqp_rt": 2, "dilqr_env_tables": 1, "dilqr_tile_cost": 2, "dilqr_tile_cost_grad": 2,
}
launch_count = 0     # running total of kernels launched through this binding
profile = None       # set to a dict {name: [(start_event, end_event), ...]} to time calls


def call(name, *args, allow=()):
    """Invoke a C-ABI entry point; counts launches and (optionally) brackets the
    call with CUDA events on the current stream for per-kernel timing.  Error codes listed
    in ``allow`` are returned instead of raised (nothing was enqueued)."""
    global launch_count
    fn = getattr(lib(), name)
    if profile is not None:
        import torch
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        profile.setdefault(name, []).append((e0, e1))
    else:
        rc = fn(*args)
    if rc in allow:
        return rc
    check(rc, name)
    launch_count += (fn_iter_launches() if name == "dilqr_mpc_iterate"
                     else KERNELS_PER_CALL.get(name, 0))
    return rc


def fn_iter_launches():
    return int(lib().dilqr_last_iterate_launches())
