"""Solve rate of the runtime-dimension LinDx kernels (DILQR_DYN_LINDX_RT) against the compiled
ones (DILQR_DYN_LINDX) on the shapes both serve, and alone on shapes without compiled kernels.

Each measurement is a 10-iteration MPC solve (the pipelined outer loop) of B problems, T = 50,
timed with CUDA events after one warm-up solve; the inputs (C alone is 50 * B * n^2 scalars)
are far larger than the 126 MB L2.  Prints one JSON line per case and writes them, with the card
name and power limit read in the same run, to argv[1] (default: lindx_rt_probe.jsonl).

    python tools/lindx_rt_probe.py [out.jsonl] [B]
"""
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sol = importlib.import_module("differentiable-ilqr_b200._solver")
lib = importlib.import_module("differentiable-ilqr_b200._lib")


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def problem(ns, nc, T, B, dtype, dev, seed=0):
    """tests/common.lindx_problem, generated on the device (the CPU generator is too slow at
    these sizes)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    n = ns + nc
    kw = dict(generator=g, device=dev, dtype=dtype)
    A = torch.randn(T, B, n, n, **kw)
    C = A.transpose(2, 3) @ A + torch.eye(n, dtype=dtype, device=dev)
    del A
    c = torch.randn(T, B, n, **kw)
    F = torch.cat((torch.eye(ns, dtype=dtype, device=dev).expand(T - 1, B, ns, ns)
                   + 0.2 * torch.randn(T - 1, B, ns, ns, **kw) / ns ** 0.5,
                   torch.randn(T - 1, B, ns, nc, **kw) / ns ** 0.5), 3)
    f = 0.1 * torch.randn(T - 1, B, ns, **kw)
    x0 = torch.randn(B, ns, **kw)
    return C, c, F, f, x0


def run(kind, ns, nc, T, B, dtype, boxed, data):
    C, c, F, f, x0 = data
    kw = dict(u_lower=-1.0, u_upper=1.0) if boxed else {}
    dyn = sol.DynSpec(kind, F=F, f=f)
    sol.solve_mpc(x0, C, c, dyn, ns, nc, T, lqr_iter=10, verbose=-1, **kw)   # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 2
    retries = 0
    e0.record()
    for _ in range(reps):
        _, _, _, info = sol.solve_mpc(x0, C, c, dyn, ns, nc, T, lqr_iter=10, verbose=-1, **kw)
        retries += info.retries
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return dict(ms_per_solve=round(ms, 3), problems_per_s=round(B / ms * 1e3),
                trace_reruns_per_solve=retries / reps, iters=info.n_iters,
                group_sweep=int(info._problem[0].group_sweep), kernels=int(info._problem[0].dynamics))


def main():
    out = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else "lindx_rt_probe.jsonl")
    B = int(sys.argv[2]) if len(sys.argv) > 2 else 65536
    T = 50
    dev = torch.device("cuda:0")
    card = device_info()
    os.makedirs(os.path.dirname(out), exist_ok=True)
    fh = open(out, "w")
    cases = [((4, 2), True), ((8, 4), True), ((16, 4), True), ((6, 1), False), ((7, 3), False),
             ((24, 8), False)]
    for dtype in (torch.float64, torch.float32):
        for (ns, nc), both in cases:
            data = problem(ns, nc, T, B, dtype, dev)
            for boxed in (False, True):
                kinds = [lib.DYN_LINDX, lib.DYN_LINDX_RT] if both else [lib.DYN_LINDX_RT]
                for kind in kinds:
                    r = dict(card=card, shape="%d+%d" % (ns, nc), dtype=str(dtype).split(".")[-1], T=T,
                             B=B, boxed=boxed,
                             path="compiled" if kind == lib.DYN_LINDX else "runtime")
                    r.update(run(kind, ns, nc, T, B, dtype, boxed, data))
                    print(json.dumps(r), flush=True)
                    fh.write(json.dumps(r) + "\n")
                    fh.flush()
            del data
            torch.cuda.empty_cache()
    fh.close()


if __name__ == "__main__":
    main()
