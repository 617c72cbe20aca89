"""Solve rate of the runtime-dimension pnqp kernels (dilqr_pnqp_rt) against the compiled ones
(dilqr_pnqp) on the sizes both serve, and alone on sizes without compiled kernels.

Each measurement is a standalone ``pnqp`` call (n_iter = 20, batch-global control flow, cold
start) of B problems H = A'A/n + I: the kernel runs until the replayed trace is confirmed, so a
call includes its trace re-runs and one status copy per run.  "free" puts the bounds at +-inf,
"boxed" draws them from U(-1, 0) / U(0, 1) so that constraints are active.  B = 65536 for
n <= 64; above, B is chosen so that H takes about 2 GB, far beyond the 126 MB L2.  Data is
generated on the device; every shape is warmed up by one call, then at least `reps` calls and
about 0.3 s of them are timed with CUDA events.  On the sizes both families serve, the outputs
of the two are compared bitwise.  Prints one JSON line per case and writes them, with the card
name and power limit read in the same run, to argv[1] (default: pnqp_rt_probe.jsonl).

    python tools/pnqp_rt_probe.py [out.jsonl] [reps]
"""
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
lib = importlib.import_module("differentiable-ilqr_b200._lib")
pm = importlib.import_module("differentiable-ilqr_b200.pnqp")


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout
    q = q.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def batch(n, dtype):
    if n <= 64:
        return 65536
    return (2 << 30) // (n * n * torch.finfo(dtype).bits // 8)


def problem(n, B, dtype, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    kw = dict(generator=g, device=dev, dtype=dtype)
    A = torch.randn(B, n, n, **kw)
    H = torch.baddbmm(torch.eye(n, dtype=dtype, device=dev).expand(B, n, n), A.transpose(1, 2), A,
                      alpha=1.0 / n)
    del A
    q = 2 * torch.randn(B, n, **kw)
    lo = -torch.rand(B, n, **kw)
    hi = torch.rand(B, n, **kw)
    return H, q, lo, hi


def timed(kind, args, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = pm.run(*args, kind=kind)          # warm-up
    e1.record()
    torch.cuda.synchronize()
    # at least `reps` calls and about 0.3 s of them
    reps = max(reps, min(200, int(300.0 / max(e0.elapsed_time(e1), 1e-3))))
    runs = 0
    e0.record()
    for _ in range(reps):
        out = pm.run(*args, kind=kind)
        runs += out[5]
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    B = args[0].shape[0]
    return out, dict(reps=reps, ms_per_call=round(ms, 3), problems_per_s=round(B / ms * 1e3),
                     trace_reruns_per_call=runs / reps - 1, qp_iters=out[3] + 1)


def same(a, b):
    fa, fb = a[1], b[1]
    fac = torch.equal(fa, fb) if torch.is_tensor(fa) else (
        torch.equal(fa[0], fb[0]) and torch.equal(fa[1], fb[1]))
    return bool(torch.equal(a[0], b[0]) and torch.equal(a[2], b[2]) and fac and a[3] == b[3])


def main():
    out = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else "pnqp_rt_probe.jsonl")
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    dev = torch.device("cuda:0")
    card = device_info()
    os.makedirs(os.path.dirname(out), exist_ok=True)
    fh = open(out, "w")
    inf = float("inf")
    for dtype in (torch.float64, torch.float32):
        for n in (2, 4, 8, 5, 16, 32, 64, 128, 256):
            B = batch(n, dtype)
            H, q, lo, hi = problem(n, B, dtype, dev)
            for boxed in (False, True):
                args = (H, q, lo, hi) if boxed else (H, q, -inf, inf)
                kinds = [lib.PNQP_COMPILED, lib.PNQP_RT] if n in (2, 4, 8) else [lib.PNQP_RT]
                results = []
                for kind in kinds:
                    o, t = timed(kind, args, reps)
                    results.append(o)
                    r = dict(card=card, n=n, dtype=str(dtype).split(".")[-1], n_iter=20, B=B,
                             boxed=boxed, path="compiled" if kind == lib.PNQP_COMPILED else "runtime")
                    r.update(t)
                    if len(results) == 2:
                        r["bitwise_equal_to_compiled"] = same(results[0], results[1])
                    print(json.dumps(r), flush=True)
                    fh.write(json.dumps(r) + "\n")
                    fh.flush()
                del results, o
            del H, q, lo, hi
            torch.cuda.empty_cache()
    fh.close()


if __name__ == "__main__":
    main()
