"""Cost of the DiLQR backward with the adjoint system solved by Richardson iteration (4 passes,
the benchmark's setting) and by restarted GMRES (restart m in {32, 64, 300}; 300 = T n is full
GMRES), cartpole T = 50, B problems (default 65536), FP64 and FP32, regimes 2a (cold start,
sigma = 0.5, 10 iLQR iterations: most problems are not at a fixed point) and 2b (sigma = 0.05,
the solve reaches its fixed point).

Per case: backward ms (CUDA events around one _solver.dilqr_backward call after a warm-up of
the same shapes; the preparation at the solution is included and is the same for every
solver), for GMRES the median / maximum Arnoldi steps per problem, the fraction of problems that
reached the tolerance within the default budget, and the peak device memory of the call.  One
JSON line per case, with the card name and power limit read in the same run, goes to argv[1]
(default: krylov_probe.jsonl).

    python tools/krylov_probe.py [out.jsonl] [B]
"""
import importlib
import json
import os
import subprocess
import sys
import warnings

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("differentiable-ilqr_b200")
sol = importlib.import_module("differentiable-ilqr_b200._solver")
env = importlib.import_module("differentiable-ilqr_b200.env_dx")

T = 50
THETA = (9.8, 1.0, 0.1, 0.5)


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout
    q = q.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def problem(B, dtype, dev, sigma):
    g = torch.Generator().manual_seed(0)
    r = (torch.rand(B, 4, generator=g, dtype=torch.float64) * 2 - 1) * sigma
    x0 = torch.stack((r[:, 0], r[:, 1], torch.cos(r[:, 2]), torch.sin(r[:, 2]), r[:, 3]), 1)
    dx = env.CartpoleDx(torch.tensor(THETA, dtype=dtype, device=dev))
    q, p = [t.to(dev, dtype) for t in dx.get_true_obj()]
    C = torch.diag(q)[None, None].expand(T, B, 6, 6).contiguous()
    c = p[None, None].expand(T, B, 6).contiguous()
    m = pkg.mpc_explicit.MPC(5, 1, T, u_lower=dx.lower, u_upper=dx.upper, lqr_iter=10,
                             eps=dx.mpc_eps, linesearch_decay=dx.linesearch_decay,
                             max_linesearch_iter=dx.max_linesearch_iter, verbose=-1,
                             exit_unconverged=False, detach_unconverged=False, n_batch=B)
    x0 = x0.to(dev, dtype)
    with torch.no_grad():
        x, u, _ = m(x0, pkg.QuadCost(C, c), dx)
    gu = torch.randn(T, B, 1, generator=torch.Generator(device=dev).manual_seed(1), device=dev,
                     dtype=dtype)
    return dx, x0, C, c, x, u, gu


def backward(data, **kw):
    dx, x0, C, c, x, u, gu = data
    stats = {}
    sol.dilqr_backward(None, gu, x0, C, c, x, u, dx, 5, 1, dx.lower, dx.upper, stats=stats, **kw)
    return stats


def timed(data, **kw):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    stats = backward(data, **kw)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), torch.cuda.max_memory_allocated() / 2 ** 30, stats


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else "krylov_probe.jsonl"
    B = int(sys.argv[2]) if len(sys.argv) > 2 else 65536
    dev = torch.device("cuda:0")
    card = device_info()
    f = open(out, "w")
    for dtype in (torch.float64, torch.float32):
        for regime, sigma in (("2a", 0.5), ("2b", 0.05)):
            data = problem(B, dtype, dev, sigma)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                backward(data, n_passes=4)                                  # warm-up
                backward(data, solver="gmres", gmres_restart=4, gmres_max_iter=4)
                cases = [("richardson", 4, dict(n_passes=4))] + [
                    ("gmres", m_, dict(solver="gmres", gmres_restart=m_)) for m_ in (32, 64, 300)]
                for name, m_, kw in cases:
                    ms, gib, st = timed(data, **kw)
                    rec = dict(solver=name, dtype=str(dtype).split(".")[-1], regime=regime, T=T,
                               B=B, backward_ms=round(ms, 2), peak_gib=round(gib, 2), card=card)
                    if name == "richardson":
                        rec.update(passes=m_, richardson_last_update_rel=st.get("resid"))
                    else:
                        gm = st["gmres"]
                        it = gm.iters.double()
                        rec.update(restart=gm.restart, max_iter=gm.max_iter, tol=gm.tol,
                                   iters_median=float(it.median()), iters_max=int(it.max()),
                                   frac_converged=round(1 - gm.unconverged / B, 6),
                                   worst_resid=gm.worst, operator_calls=gm.op_calls)
                    print(json.dumps(rec), flush=True)
                    f.write(json.dumps(rec) + "\n")
                    f.flush()
            del data
            torch.cuda.empty_cache()
    f.close()


if __name__ == "__main__":
    main()
