"""Solve rate of the runtime-dimension network kernels (DILQR_DYN_NN_RT) against the compiled
ones (DILQR_DYN_NN) on the shapes both serve, and alone on shapes without compiled kernels.

The dynamics are an NNDynamics with one sigmoid hidden layer of H units (passthrough, analytic
linearisation).  Each measurement is one 10-iteration MPC solve (the pipelined outer loop) of B
problems, T = 50, timed with CUDA events after a warm-up solve of the same shape on 256 problems;
the cost inputs (C alone is 50 * B * n^2 scalars) are far larger than the 126 MB L2.  Prints one
JSON line per case and writes them, with the card name and power limit read in the same run, to
argv[1] (default: nn_rt_probe.jsonl).

    python tools/nn_rt_probe.py [out.jsonl] [B]
"""
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
dilqr = importlib.import_module("differentiable-ilqr_b200")
sol = importlib.import_module("differentiable-ilqr_b200._solver")
lib = importlib.import_module("differentiable-ilqr_b200._lib")


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def problem(ns, nc, T, B, dtype, dev, seed=0):
    """The cost and initial states of tests/common.lindx_problem, generated on the device."""
    g = torch.Generator(device=dev).manual_seed(seed)
    n = ns + nc
    kw = dict(generator=g, device=dev, dtype=dtype)
    A = torch.randn(T, B, n, n, **kw)
    C = A.transpose(2, 3) @ A + torch.eye(n, dtype=dtype, device=dev)
    del A
    c = torch.randn(T, B, n, **kw)
    x0 = torch.randn(B, ns, **kw)
    return C, c, x0


def network(ns, nc, H, dtype, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    net = dilqr.NNDynamics(ns, nc, hidden_sizes=[H], activation="sigmoid").double()
    with torch.no_grad():
        for fc in net.fcs:
            fc.weight.copy_(torch.randn(fc.weight.shape, generator=g, dtype=torch.float64)
                            / fc.weight.shape[1] ** 0.5)
            fc.bias.copy_(0.1 * torch.randn(fc.bias.shape, generator=g, dtype=torch.float64))
        net.fcs[-1].weight.mul_(0.3)
    return net._dilqr_pack(dtype, dev)


def run(kind, ns, nc, T, B, dtype, boxed, data, pack):
    C, c, x0 = data
    kw = dict(u_lower=-1.0, u_upper=1.0) if boxed else {}
    dyn = sol.DynSpec(kind, aux=pack[0], ai=pack[1])
    w = 256   # warm-up: module load and the workspace of this shape
    sol.solve_mpc(x0[:w], C[:, :w], c[:, :w], dyn, ns, nc, T, lqr_iter=10, verbose=-1, **kw)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _, _, _, info = sol.solve_mpc(x0, C, c, dyn, ns, nc, T, lqr_iter=10, verbose=-1, **kw)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return dict(ms_per_solve=round(ms, 3), problems_per_s=round(B / ms * 1e3),
                trace_reruns_per_solve=info.retries, iters=info.n_iters,
                kernels=int(info._problem[0].dynamics))


def main():
    out = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else "nn_rt_probe.jsonl")
    B = int(sys.argv[2]) if len(sys.argv) > 2 else 65536
    T = 50
    dev = torch.device("cuda:0")
    card = device_info()
    os.makedirs(os.path.dirname(out), exist_ok=True)
    fh = open(out, "w")
    cases = [((3, 1), 32, True), ((4, 2), 32, True), ((5, 1), 32, True)]
    cases += [((ns, nc), H, False) for ns, nc in ((6, 2), (12, 4), (24, 8)) for H in (32, 128)]
    for dtype in (torch.float64, torch.float32):
        for (ns, nc), H, both in cases:
            data = problem(ns, nc, T, B, dtype, dev)
            pack = network(ns, nc, H, dtype, dev)
            for boxed in (False, True):
                kinds = [lib.DYN_NN, lib.DYN_NN_RT] if both else [lib.DYN_NN_RT]
                for kind in kinds:
                    r = dict(card=card, shape="%d+%d" % (ns, nc), H=H, dtype=str(dtype).split(".")[-1],
                             T=T, B=B, boxed=boxed, path="compiled" if kind == lib.DYN_NN else "runtime")
                    r.update(run(kind, ns, nc, T, B, dtype, boxed, data, pack))
                    print(json.dumps(r), flush=True)
                    fh.write(json.dumps(r) + "\n")
                    fh.flush()
            del data
            torch.cuda.empty_cache()
    fh.close()


if __name__ == "__main__":
    main()
